// rfm_kernels.cu -- hand-written sm_100a kernels for the IQ -> audio (+RDS) chain.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo ...
// All arithmetic that feeds the reference's rounding-sensitive recurrences goes through the
// individually rounded helpers of rfm_math.cuh in the reference's operation order, so the
// results are bit-identical to the CPU chain (see DESIGN.md, "Numerics").
//
// Kernel map (SURVEY.md section 7 / 8a rows in brackets):
//   k_front        [a1 a3 a5]   u8 | s8 | s16 | cf32 -> float -> fine-tuner rotate -> Lanczos FIR / ds; tile of outputs
//                               per CTA, input + halo staged in shared memory
//   k_front_tail   [a5 state]   last `order` tuned samples -> m_stateComplex
//   k_bb_lanes     [a4 a6 a13 a15 a16] one lane per stream: IF meter, FM-demod PLL + DC tracker,
//                               baseband meters, 19 kHz pilot PLL, 38 kHz demux multiply
//   k_resample     [a14 x2]     fractional Lanczos resampler, mono + stereo share taps
//   k_rotfir       [a8 a10 a17] cFirFilter (rotating summation start), real / pair / complex
//   k_audio_tail   [a18 a19 a20] deemphasis + notch + L/R matrix, one lane per stream
//   k_osc          [a7 NCO]     quadrature-oscillator table for the block (same for every stream)
//   k_rds_front    [a7 a8]      NCO mix + every decimate-by-2 stage + RDS LP, fused in shared memory
//   k_rds_pll      [a9]         Costas loop, one lane per stream
//   k_rds_slice    [a11]        bit-clock resonator + peak slicer + differential decode
//   k_tails                     V-buffer history carry
#include <cuda.h> // CUtensorMap (declarations only: the encoder is looked up at run time, libcuda is not linked)

#include "rfm_kernels.cuh"
#include "rfm_dsp.cuh"

#include <assert.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <utility>

namespace rfm
{

static inline unsigned cdiv(unsigned a, unsigned b) { return (a + b - 1) / b; }

void EnsureDynSmemImpl(const void* func, size_t smem)
{
  static std::mutex mu;
  static std::map<std::pair<int, const void*>, size_t> set;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = set[std::make_pair(dev, func)];
  if (smem > cur)
  {
    cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cur = smem;
  }
}

// ==================================================================================================
// front end
// ==================================================================================================
constexpr unsigned kFrontTile = 128; // outputs per CTA == threads per CTA

// fine-tuned sample i of this block: (IQ format F -> float) * table[(idx0 + i) mod 64]
// RTL_SDR_Source.cpp:207-211, FmDecode.cpp:66-82 (std::complex product: ac-bd, ad+bc)
template <int F>
__device__ __forceinline__ float2 tuned_sample(const void* __restrict__ row, unsigned i, unsigned idx0,
                                               const float* lut, const float2* tuner)
{
  float are, aim;
  if (F == kIqU8)
  {
    const uchar2 u = reinterpret_cast<const uchar2*>(row)[i];
    are = lut[u.x];
    aim = lut[u.y];
  }
  else if (F == kIqS8)
  {
    const unsigned w = reinterpret_cast<const unsigned short*>(row)[i];
    are = rfm_s8_to_float(w, 0u);
    aim = rfm_s8_to_float(w, 1u);
  }
  else if (F == kIqS16)
  {
    const unsigned w = reinterpret_cast<const unsigned*>(row)[i];
    are = rfm_s16_to_float(w, 0u);
    aim = rfm_s16_to_float(w, 1u);
  }
  else
  {
    const float2 f = reinterpret_cast<const float2*>(row)[i];
    are = f.x;
    aim = f.y;
  }
  if (!tuner) // stand-alone cDownsampleFilter (rfm_downsample): no fine tuner in front of the FIR
    return make_float2(are, aim);
  const float2 b = tuner[(idx0 + i) & 63u];
  float2 o;
  o.x = subf(mulf(are, b.x), mulf(aim, b.y));
  o.y = addf(mulf(are, b.y), mulf(aim, b.x));
  return o;
}

template <int F>
__global__ void __launch_bounds__(kFrontTile) k_front(FrontParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_lut = reinterpret_cast<float*>(smem_raw);
  float2* s_tuner = reinterpret_cast<float2*>(s_lut + 256);
  float* s_coef = reinterpret_cast<float*>(s_tuner + 64);
  const unsigned coef_n = (p.order + 2 + 1) & ~1u;
  float2* X = reinterpret_cast<float2*>(s_coef + coef_n);

  const unsigned tid = threadIdx.x;
  const unsigned s = blockIdx.y;
  const unsigned o0 = blockIdx.x * kFrontTile;
  const unsigned nt = min(kFrontTile, p.nout - o0);

  for (unsigned i = tid; i < 256; i += kFrontTile)
    s_lut[i] = p.lut[i];
  if (tid < 64)
    s_tuner[tid] = p.tuner ? reinterpret_cast<const float2*>(p.tuner)[tid] : make_float2(0.f, 0.f);
  for (unsigned i = tid; i < p.order + 2; i += kFrontTile)
    s_coef[i] = p.coeff[i];
  __syncthreads();

  // V = tail(order) ++ block(n); this tile needs V[vlo .. vlo + count)
  const unsigned vlo = p.p0 + o0 * p.ds;
  const unsigned count = (nt - 1) * p.ds + p.order;
  const size_t esz = IqBytes(F);
  const unsigned char* row = reinterpret_cast<const unsigned char*>(p.in) + (size_t)s * p.in_stride * esz;
  const float2* tail = reinterpret_cast<const float2*>(p.tail) + (size_t)s * p.order;
  for (unsigned v = tid; v < count; v += kFrontTile)
  {
    const unsigned V = vlo + v;
    X[v] = (V < p.order) ? tail[V] : tuned_sample<F>(row, V - p.order, p.idx0, s_lut, p.tuner ? s_tuner : nullptr);
  }
  __syncthreads();

  if (tid < nt)
  {
    // y = sum_{j=1..order} x[p - j] * c[j], ascending j, complex x real (DownConvert.cpp:112-129)
    const float2* xp = X + tid * p.ds + p.order;
    float yr = 0.0f, yi = 0.0f;
    for (unsigned j = 1; j <= p.order; ++j)
    {
      const float2 x = xp[-(int)j];
      const float c = s_coef[j];
      yr = addf(yr, mulf(x.x, c));
      yi = addf(yi, mulf(x.y, c));
    }
    reinterpret_cast<float2*>(p.z)[(size_t)s * p.z_stride + o0 + tid] = make_float2(yr, yi);
  }
}

template <int F>
__global__ void __launch_bounds__(256) k_front_tail(FrontParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* tmp = reinterpret_cast<float2*>(smem_raw);
  const unsigned s = blockIdx.x;
  const size_t esz = IqBytes(F);
  const unsigned char* row = reinterpret_cast<const unsigned char*>(p.in) + (size_t)s * p.in_stride * esz;
  float2* tail = reinterpret_cast<float2*>(p.tail) + (size_t)s * p.order;
  const float2* tuner = reinterpret_cast<const float2*>(p.tuner);
  for (unsigned k = threadIdx.x; k < p.order; k += blockDim.x)
  {
    const unsigned V = p.n + k; // new tail = V[n .. n + order)
    tmp[k] = (V < p.order) ? tail[V] : tuned_sample<F>(row, V - p.order, p.idx0, p.lut, tuner);
  }
  __syncthreads();
  for (unsigned k = threadIdx.x; k < p.order; k += blockDim.x)
    tail[k] = tmp[k];
}

// --------------------------------------------------------------------------------------------------
// Register-tiled front end for the decimations the reference's caller produces (ds = 1, 4, 5, 11; order = 8 ds).
//   * a CTA of 128 threads makes 512 consecutive outputs of one stream; every thread owns R = 4 consecutive outputs;
//   * the tuned input window ((512-1) ds + order samples) is formed once in shared memory.  u8 -> float uses the
//     exact two-FMA form of the reference's double expression (rfm_u8_to_float, all 256 codes checked), so no
//     table lookups; the 8 fine-tuner phasors a thread needs are loop-invariant registers;
//   * the FIR walks the thread's window from the newest sample down: each sample is loaded ONCE (LDS.64) and feeds
//     up to R accumulators, each of which therefore receives its taps in ascending j -- the reference's
//     summation order (DownConvert.cpp:112-129); products and sums are individually rounded (no FMA);
//   * taps come from the kernel-parameter constant bank with compile-time offsets (no loads);
//   * the window is stored with one padding slot per R*ds samples: thread stride R*ds+1 (odd) float2 ->
//     conflict-free 64-bit shared loads.
// --------------------------------------------------------------------------------------------------
struct FrontCoef
{
  float c[92]; // c[j], j = 0 .. order + 1 (order <= 88)
};

template <int DS>
struct FrontGeom
{
  static constexpr int R = 4, T = 128, ORDER = 8 * DS, OB = T * R, SEG = R * DS;
  static constexpr int W = (OB - 1) * DS + ORDER;          // window samples
  static constexpr int WIN = ORDER + DS * (R - 1);         // samples one thread touches
  static constexpr int WP = W + (W - 1) / SEG + 1;         // padded window
  __host__ __device__ static constexpr int pos(int w) { return w + w / SEG; }
};

// BYTES: two-byte samples (u8, s8) staged in 16-byte chunks, else one load per sample (s16, cf32); F: IqFormat
template <bool BYTES, int DS, int F = BYTES ? kIqU8 : kIqCF32>
__global__ void __launch_bounds__(128) k_front_tiled(FrontParams p, FrontCoef cf)
{
  using G = FrontGeom<DS>;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* X = reinterpret_cast<float2*>(smem_raw);

  const unsigned tid = threadIdx.x;
  const unsigned s = blockIdx.y;
  const unsigned o0 = blockIdx.x * G::OB;
  const unsigned nt = min((unsigned)G::OB, p.nout - o0);
  // V = tail(order) ++ block(n); this CTA needs V[vlo .. vlo + count)
  const unsigned vlo = p.p0 + o0 * DS;
  const unsigned count = (nt - 1) * DS + G::ORDER;
  const float2* tuner = reinterpret_cast<const float2*>(p.tuner);

  // ---- window: history part (first CTA of a row only)
  if (vlo < (unsigned)G::ORDER)
  {
    const float2* tail = reinterpret_cast<const float2*>(p.tail) + (size_t)s * G::ORDER;
    for (unsigned V = vlo + tid; V < (unsigned)G::ORDER && V - vlo < count; V += G::T)
      X[G::pos((int)(V - vlo))] = tail[V];
  }
  // ---- window: new samples i in [i_lo, i_hi) of this block, sample i lands at w = i + order - vlo
  const int i_lo = max(0, (int)vlo - G::ORDER);
  const int i_hi = min((int)p.n, (int)(vlo + count) - G::ORDER);
  static_assert(BYTES == (F == kIqU8 || F == kIqS8), "staging follows the sample size");
  if (BYTES)
  {
    const unsigned char* row = reinterpret_cast<const unsigned char*>(p.in) + (size_t)s * p.in_stride * 2;
    // 16-byte chunks of 8 samples, aligned in memory: chunk c holds samples k0 + 8c .. k0 + 8c + 7
    const int k0 = (int)(((16u - (unsigned)(reinterpret_cast<uintptr_t>(row) & 15u)) & 15u) >> 1);
    const int c_lo = (i_lo - k0) >= 0 ? (i_lo - k0) / 8 : -(((k0 - i_lo) + 7) / 8);
    // a thread's chunks are 128 chunks = 1024 samples apart: its 8 tuner phasors never change
    float2 tw[8];
    const int ib0 = k0 + 8 * (c_lo + (int)tid);
#pragma unroll
    for (int e = 0; e < 8; ++e)
      tw[e] = tuner[(p.idx0 + (unsigned)(ib0 + e)) & 63u];
    // (kept as a rolled loop: the unrolled FIR below already fills most of the 32 KB instruction cache; the 16-byte
    // load of the NEXT interior chunk is issued before the current one is converted)
    auto interior = [&](int ib) { return ib >= i_lo && ib + 8 <= i_hi; };
    uint4 nxt = make_uint4(0u, 0u, 0u, 0u);
    if (interior(ib0))
      nxt = *reinterpret_cast<const uint4*>(row + 2 * (size_t)ib0);
#pragma unroll 1
    for (int ib = ib0; ib < i_hi; ib += 8 * G::T)
    {
      const uint4 cur = nxt;
      const int ibn = ib + 8 * G::T;
      if (ibn < i_hi && interior(ibn))
        nxt = *reinterpret_cast<const uint4*>(row + 2 * (size_t)ibn);
      if (interior(ib))
      {
        // interior chunk (the common case): one 16-byte load, no per-sample predicates
        const uint4 raw = cur;
        const unsigned wd[4] = {raw.x, raw.y, raw.z, raw.w};
        const int w0 = ib + G::ORDER - (int)vlo;
        const int q0 = w0 / G::SEG, rem = w0 - q0 * G::SEG;
        float2* xo = X + w0 + q0;
#pragma unroll
        for (int e = 0; e < 8; ++e)
        {
          const unsigned word = wd[e >> 1];
          const float are = rfm_iq8_to_float<F>(word, (e & 1) ? 2u : 0u);
          const float aim = rfm_iq8_to_float<F>(word, (e & 1) ? 3u : 1u);
          float2 o;
          o.x = subf(mulf(are, tw[e].x), mulf(aim, tw[e].y));   // FmDecode.cpp:66-82
          o.y = addf(mulf(are, tw[e].y), mulf(aim, tw[e].x));
          const int carry = (G::SEG >= 8) ? ((rem + e >= G::SEG) ? 1 : 0) : (rem + e) / G::SEG;
          xo[e + carry] = o;
        }
        continue;
      }
      uint4 raw;
      if (ib >= 0 && ib + 8 <= (int)p.n)
        raw = *reinterpret_cast<const uint4*>(row + 2 * (size_t)ib);
      else
      {
        unsigned short h[8];
#pragma unroll
        for (int e = 0; e < 8; ++e)
          h[e] = (ib + e >= 0 && ib + e < (int)p.n) ? *reinterpret_cast<const unsigned short*>(row + 2 * (size_t)(ib + e)) : (unsigned short)0;
        raw.x = h[0] | ((unsigned)h[1] << 16); raw.y = h[2] | ((unsigned)h[3] << 16);
        raw.z = h[4] | ((unsigned)h[5] << 16); raw.w = h[6] | ((unsigned)h[7] << 16);
      }
      const unsigned wd[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
      for (int e = 0; e < 8; ++e)
      {
        const int i = ib + e;
        if (i >= i_lo && i < i_hi)
        {
          const unsigned word = wd[e >> 1];
          const float are = rfm_iq8_to_float<F>(word, (e & 1) ? 2u : 0u);
          const float aim = rfm_iq8_to_float<F>(word, (e & 1) ? 3u : 1u);
          float2 o;
          o.x = subf(mulf(are, tw[e].x), mulf(aim, tw[e].y));
          o.y = addf(mulf(are, tw[e].y), mulf(aim, tw[e].x));
          X[G::pos(i + G::ORDER - (int)vlo)] = o;
        }
      }
    }
  }
  else if (F == kIqS16)
  {
    // one 32-bit word per sample: the rows are read as the cf32 rows below, half the bytes
    const unsigned* row = reinterpret_cast<const unsigned*>(p.in) + (size_t)s * p.in_stride;
    for (int i = i_lo + (int)tid; i < i_hi; i += G::T)
    {
      const unsigned w = row[i];
      const float2 a = make_float2(rfm_s16_to_float(w, 0u), rfm_s16_to_float(w, 1u));
      const float2 b = tuner[(p.idx0 + (unsigned)i) & 63u];
      float2 o;
      o.x = subf(mulf(a.x, b.x), mulf(a.y, b.y));
      o.y = addf(mulf(a.x, b.y), mulf(a.y, b.x));
      X[G::pos(i + G::ORDER - (int)vlo)] = o;
    }
  }
  else
  {
    const float2* row = reinterpret_cast<const float2*>(p.in) + (size_t)s * p.in_stride;
    for (int i = i_lo + (int)tid; i < i_hi; i += G::T)
    {
      const float2 a = row[i];
      const float2 b = tuner[(p.idx0 + (unsigned)i) & 63u];
      float2 o;
      o.x = subf(mulf(a.x, b.x), mulf(a.y, b.y));
      o.y = addf(mulf(a.x, b.y), mulf(a.y, b.x));
      X[G::pos(i + G::ORDER - (int)vlo)] = o;
    }
  }
  __syncthreads();

  // ---- FIR: outputs tid*R .. tid*R + R-1; thread window w = SEG*tid + (WIN-1) - u, u = 0 .. WIN-1 (newest first)
  if (tid * G::R >= nt)
    return;
  float2 acc[G::R];
#pragma unroll
  for (int i = 0; i < G::R; ++i)
    acc[i] = make_float2(0.0f, 0.0f);
  const float2* xt = X + tid * (G::SEG + 1);
#pragma unroll
  for (int u = 0; u < G::WIN; ++u)
  {
    const int wl = G::WIN - 1 - u; // local window index; pos(SEG*tid + wl) = (SEG+1)*tid + wl + wl/SEG
    const float2 v = xt[wl + wl / G::SEG];
#pragma unroll
    for (int i = 0; i < G::R; ++i)
    {
      const int j = u + 1 - DS * (G::R - 1 - i); // tap of output i that meets this sample
      if (j >= 1 && j <= G::ORDER)
      {
        acc[i].x = addf(acc[i].x, mulf(v.x, cf.c[j]));
        acc[i].y = addf(acc[i].y, mulf(v.y, cf.c[j]));
      }
    }
  }
  float2* zo = reinterpret_cast<float2*>(p.z) + (size_t)s * p.z_stride + o0 + tid * G::R;
  if (tid * G::R + G::R <= nt)
  {
    reinterpret_cast<float4*>(zo)[0] = make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y);
    reinterpret_cast<float4*>(zo)[1] = make_float4(acc[2].x, acc[2].y, acc[3].x, acc[3].y);
  }
  else
  {
#pragma unroll
    for (int i = 0; i < G::R; ++i)
      if (tid * G::R + i < nt)
        zo[i] = acc[i];
  }
}

// --------------------------------------------------------------------------------------------------
// TMA form of the same kernel for u8 and s8 input (same byte geometry) and ds = 1, 5, 11 (390 625 S/s, 1.2, 2.4 MS/s).
//   * the raw u8 window -- ((384-1) ds + order) IQ pairs plus alignment -- is fetched by the TMA unit: one elected
//     thread issues cp.async.bulk.tensor.2d over a tensor map of the caller's [S][n] rows (8-byte elements = 4 IQ
//     pairs, boxes of 256 elements = 2 KB) and the CTA waits on an mbarrier.  Out-of-range coordinates (before the
//     row: the history part comes from the tail buffer; behind it) are zero-filled by the hardware: no edge paths,
//     no per-sample predicates, no address arithmetic in the conversion loop;
//   * the raw bytes land at the END of the window buffer they are expanded into; every thread pulls its 16-byte
//     chunks into registers, one barrier retires the raw region, then u8 -> float -> fine tuner -> window as before;
//   * R = 3 outputs per thread: the thread stride R ds float2 = 6 ds words is 2 (mod 4) banks for odd ds, so the
//     64-bit window loads of a half warp are conflict-free WITHOUT the padding slot of the R = 4 kernel -- and with
//     it goes the carry logic of the staging stores (4 of its 24 instructions per sample).  Six CTAs per SM.
// Same taps, same products, same ascending-j summation per output (DownConvert.cpp:112-129).
// --------------------------------------------------------------------------------------------------
template <int DS>
struct FrontGeom3
{
  static constexpr int R = 3, T = 128, ORDER = 8 * DS, OB = T * R, SEG = R * DS;
  static constexpr int W = (OB - 1) * DS + ORDER;          // window samples
  static constexpr int WIN = ORDER + DS * (R - 1);         // samples one thread touches
  static constexpr int RAW_ELEMS = (W + 7 + 3) / 4 + 1;    // 8-byte elements that cover any alignment of the window (a box
                                                           // must start on a 16-byte boundary of global memory: 8 IQ pairs)
  static constexpr int BOXES = (RAW_ELEMS + 255) / 256;    // 2 KB boxes
  static constexpr int NPAIR = (BOXES * 512 + T - 1) / T;  // IQ pairs of pairs (32-bit words) per thread
  static constexpr int XBYTES = (W + 1) * 8;               // + 1: the window is shifted by one slot when vlo is odd
  // the raw window has its own region behind the float window: it is refilled (next tile) while this one is filtered
  static constexpr int RAW_OFF = (XBYTES + 127) / 128 * 128;
  static constexpr int SMEM = RAW_OFF + BOXES * 2048;
  static_assert(RAW_OFF >= ORDER * 8 && RAW_OFF % 128 == 0, "raw region must not overlap the history part of the window");
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

template <int F, int DS, bool FUSED>
__device__ __forceinline__ void front_tma(const FrontParams& p, const FrontCoef& cf, const CUtensorMap& tmap,
                                          unsigned tiles_per_row, unsigned total_tiles)
{
  using G = FrontGeom3<DS>;
  extern __shared__ __align__(128) unsigned char smem_front_tma[];
  __shared__ __align__(8) unsigned long long mbar;
  float2* X = reinterpret_cast<float2*>(smem_front_tma);
  const unsigned char* raw = smem_front_tma + G::RAW_OFF;

  const unsigned tid = threadIdx.x;
  const float2* tuner = reinterpret_cast<const float2*>(p.tuner);
  // persistent CTA: tiles blockIdx.x, blockIdx.x + gridDim.x, ...; the TMA fetch of the NEXT tile's raw window is in
  // flight while this tile is converted and filtered
  auto issue = [&](unsigned tile) {
    const unsigned s = tile / tiles_per_row, bx = tile - s * tiles_per_row;
    // first 8-byte element: the window start rounded down to 8 IQ pairs (16 bytes -- the TMA unit faults on a box whose
    // first byte is not 16-byte aligned); negative at a row's start
    const int c0 = (((int)(p.p0 + bx * G::OB * DS) - G::ORDER) >> 3) * 2;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&mbar)), "r"(G::BOXES * 2048) : "memory");
#pragma unroll
    for (int b = 0; b < G::BOXES; ++b)
      asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                   ::"r"(smem_u32(raw + b * 2048)), "l"(reinterpret_cast<unsigned long long>(&tmap)), "r"(smem_u32(&mbar)),
                   "r"(c0 + 256 * b), "r"((int)s)
                   : "memory");
  };
  if (tid == 0)
  {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&mbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (blockIdx.x < total_tiles)
      issue(blockIdx.x);
  }
  __syncthreads();
  unsigned phase = 0;
  for (unsigned tile = blockIdx.x; tile < total_tiles; tile += gridDim.x)
  {
    const unsigned s = tile / tiles_per_row, bx = tile - s * tiles_per_row;
    const unsigned o0 = bx * G::OB;
    const unsigned nt = min((unsigned)G::OB, p.nout - o0);
    // V = tail(order) ++ block(n); this tile needs V[vlo .. vlo + count)
    const int vlo = (int)(p.p0 + o0 * DS);
    const int count = (int)(nt - 1) * DS + G::ORDER;
    const int i_lo = max(0, vlo - G::ORDER);                       // block samples [i_lo, i_hi) -> w = i + order - vlo
    const int i_hi = min((int)p.n, vlo + count - G::ORDER);
    const int c0 = ((vlo - G::ORDER) >> 3) * 2;
    // A thread converts the IQ pairs 2 m, 2 m + 1 (counted from the raw window's first pair), m = tid + 128 j: one
    // 32-bit load, one 16-byte store per pair -- consecutive lanes touch consecutive words / quads of shared memory, so
    // neither side has bank conflicts (8 consecutive pairs per lane made the window stores collide 8-way: 120 M
    // conflict wavefronts per launch).  Its pairs are 256 samples apart: the two fine-tuner phasors never change.
    const int ib0 = 4 * c0 + 2 * (int)tid;
    const float2 tw0 = tuner[(p.idx0 + (unsigned)ib0) & 63u], tw1 = tuner[(p.idx0 + (unsigned)(ib0 + 1)) & 63u];
    // window slot of sample i: i + order - vlo (+ 1 when vlo is odd, so that even i lands on a 16-byte boundary)
    float2* Xs = X + (vlo & 1);
    {
      unsigned done = 0;
      while (!done)
        asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2; selp.u32 %0, 1, 0, q; }"
                     : "=r"(done) : "r"(smem_u32(&mbar)), "r"(phase) : "memory");
      phase ^= 1u;
    }
    __syncthreads(); // every thread has left the previous tile's FIR: X may be rewritten
    // ---- window: history part (first tile of a row only)
    if (vlo < G::ORDER)
    {
      const float2* tail = reinterpret_cast<const float2*>(p.tail) + (size_t)s * G::ORDER;
      for (int V = vlo + (int)tid; V < G::ORDER && V - vlo < count; V += G::T)
        Xs[V - vlo] = tail[V];
    }
    const unsigned* raw32 = reinterpret_cast<const unsigned*>(raw) + tid;
    auto tuned_pair = [&](int j) {
      const unsigned word = raw32[G::T * j];
      const float are0 = rfm_iq8_to_float<F>(word, 0u), aim0 = rfm_iq8_to_float<F>(word, 1u);
      const float are1 = rfm_iq8_to_float<F>(word, 2u), aim1 = rfm_iq8_to_float<F>(word, 3u);
      float4 o;
      o.x = subf(mulf(are0, tw0.x), mulf(aim0, tw0.y));   // FmDecode.cpp:66-82
      o.y = addf(mulf(are0, tw0.y), mulf(aim0, tw0.x));
      o.z = subf(mulf(are1, tw1.x), mulf(aim1, tw1.y));
      o.w = addf(mulf(are1, tw1.y), mulf(aim1, tw1.x));
      return o;
    };
    float2* xw = Xs + (ib0 + G::ORDER - vlo); // slot of this thread's pair j = 0; pair j is 2 T slots further
    {
      // pairs that lie completely inside [i_lo, i_hi): no predicates (sample index of pair j: ib0 + 256 j)
      const int jA = max(0, (i_lo - ib0 + 2 * G::T - 1) >> 8);
      const int jB = (i_hi - 2 - ib0) >= 0 ? ((i_hi - 2 - ib0) >> 8) + 1 : 0;
      static_assert(2 * G::T == 256, "pair stride");
#pragma unroll 4
      for (int j = jA; j < jB; ++j)
        *reinterpret_cast<float4*>(xw + 2 * G::T * j) = tuned_pair(j);
      // the (at most two) pairs of a window that straddle its ends
      const int dl = i_lo - 1 - ib0, dh = i_hi - 1 - ib0;
      if (dl >= 0 && (dl & 255) == 0 && i_lo < i_hi)
      {
        const float4 o = tuned_pair(dl >> 8);
        xw[2 * G::T * (dl >> 8) + 1] = make_float2(o.z, o.w);
      }
      if (dh >= 0 && (dh & 255) == 0 && i_hi - 1 >= i_lo)
      {
        const float4 o = tuned_pair(dh >> 8);
        xw[2 * G::T * (dh >> 8)] = make_float2(o.x, o.y);
      }
    }
    __syncthreads();
    // the raw window has gone through the conversion: its region may be refilled.  The next tile's fetch overlaps the
    // FIR below.
    if (tid == 0 && tile + gridDim.x < total_tiles)
    {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // generic-proxy reads before the async-proxy writes
      issue(tile + gridDim.x);
    }

    // ---- FIR: outputs tid*R .. tid*R + R-1; thread window w = SEG*tid + (WIN-1) - u, u = 0 .. WIN-1 (newest first)
    if (tid * G::R < nt)
    {
      float2 acc[G::R];
#pragma unroll
      for (int i = 0; i < G::R; ++i)
        acc[i] = make_float2(0.0f, 0.0f);
      const float2* xt = Xs + tid * G::SEG;
#pragma unroll
      for (int u = 0; u < G::WIN; ++u)
      {
        const float2 v = xt[G::WIN - 1 - u];
#pragma unroll
        for (int i = 0; i < G::R; ++i)
        {
          const int j = u + 1 - DS * (G::R - 1 - i); // tap of output i that meets this sample
          if (j >= 1 && j <= G::ORDER)
          {
            acc[i].x = macf<FUSED>(acc[i].x, v.x, cf.c[j]);
            acc[i].y = macf<FUSED>(acc[i].y, v.y, cf.c[j]);
          }
        }
      }
      float2* zo = reinterpret_cast<float2*>(p.z) + (size_t)s * p.z_stride + o0 + tid * G::R;
#pragma unroll
      for (int i = 0; i < G::R; ++i)
        if (tid * G::R + i < nt)
          zo[i] = acc[i];
    }
  }
}

// u8 and s8 share the byte geometry (tensor map, boxes, pair-per-lane staging); only the conversion of a pair differs
template <int DS, bool FUSED>
__global__ void __launch_bounds__(128) k_front_tma(FrontParams p, FrontCoef cf, const __grid_constant__ CUtensorMap tmap,
                                                   unsigned tiles_per_row, unsigned total_tiles)
{
  front_tma<kIqU8, DS, FUSED>(p, cf, tmap, tiles_per_row, total_tiles);
}
template <int DS, bool FUSED>
__global__ void __launch_bounds__(128) k_front_cs8_tma(FrontParams p, FrontCoef cf, const __grid_constant__ CUtensorMap tmap,
                                                       unsigned tiles_per_row, unsigned total_tiles)
{
  front_tma<kIqS8, DS, FUSED>(p, cf, tmap, tiles_per_row, total_tiles);
}
template <int F, int DS, bool FUSED>
static constexpr auto front_tma_kernel() { return F == kIqS8 ? k_front_cs8_tma<DS, FUSED> : k_front_tma<DS, FUSED>; }

// cuTensorMapEncodeTiled through the runtime's driver entry point (libcuda is not linked)
static bool EncodeFrontMap(const FrontParams& p, CUtensorMap* map)
{
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
    {
      cudaGetLastError();
      f = nullptr;
    }
    return reinterpret_cast<EncodeFn>(f);
  }();
  if (!fn)
    return false;
  const cuuint64_t dims[2] = {p.n / 4, p.S};                      // 8-byte elements = 4 IQ pairs
  const cuuint64_t strides[1] = {(cuuint64_t)p.in_stride * 2};    // bytes between rows
  const cuuint32_t box[2] = {256, 1};
  const cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void*>(p.in), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int F, int DS, bool FUSED>
static bool launch_front_tma(const FrontParams& p, const FrontCoef& cf, cudaStream_t st)
{
  using G = FrontGeom3<DS>;
  CUtensorMap map;
  if (!EncodeFrontMap(p, &map))
    return false;
  const auto kernel = front_tma_kernel<F, DS, FUSED>();
  EnsureDynSmem(kernel, G::SMEM);
  const unsigned tpr = cdiv(p.nout, G::OB), total = tpr * p.S;
  // persistent: one wave of resident CTAs (as many as fit on the device), each walks total / grid tiles
  int dev = 0, sms = 0, occ = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (p.sm_count) // the launching stream lives in an SM partition
    sms = (int)p.sm_count;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, G::T, G::SMEM) != cudaSuccess)
    occ = 1;
  const unsigned grid = std::min<unsigned>(total, (unsigned)(std::max(sms, 1) * std::max(occ, 1)));
  kernel<<<grid, G::T, G::SMEM, st>>>(p, cf, map, tpr, total);
  return true;
}

template <int F, int DS>
static void launch_front_tiled(const FrontParams& p, const FrontCoef& cf, cudaStream_t st)
{
  using G = FrontGeom<DS>;
  constexpr bool kBytes = F == kIqU8 || F == kIqS8;
  const size_t smem = (size_t)G::WP * sizeof(float2);
  EnsureDynSmem(k_front_tiled<kBytes, DS, F>, smem);
  dim3 grid(cdiv(p.nout, G::OB), p.S);
  k_front_tiled<kBytes, DS, F><<<grid, G::T, smem, st>>>(p, cf);
}

template <int F>
static bool launch_front_tma_ds(const FrontParams& p, const FrontCoef& cf, cudaStream_t st)
{
  if (p.fused)
    return p.ds == 11 ? launch_front_tma<F, 11, true>(p, cf, st) : p.ds == 5 ? launch_front_tma<F, 5, true>(p, cf, st) : launch_front_tma<F, 1, true>(p, cf, st);
  return p.ds == 11 ? launch_front_tma<F, 11, false>(p, cf, st) : p.ds == 5 ? launch_front_tma<F, 5, false>(p, cf, st) : launch_front_tma<F, 1, false>(p, cf, st);
}

template <int F>
static void launch_front_tiled_ds(const FrontParams& p, const FrontCoef& cf, cudaStream_t st)
{
  switch (p.ds)
  {
    case 1: launch_front_tiled<F, 1>(p, cf, st); break;
    case 4: launch_front_tiled<F, 4>(p, cf, st); break;
    case 5: launch_front_tiled<F, 5>(p, cf, st); break;
    default: launch_front_tiled<F, 11>(p, cf, st); break;
  }
}

template <int F>
static void launch_front_generic(const FrontParams& p, cudaStream_t st)
{
  const unsigned coef_n = (p.order + 2 + 1) & ~1u;
  const size_t smem = (256 + 128 + coef_n) * sizeof(float) + ((size_t)(kFrontTile - 1) * p.ds + p.order) * sizeof(float2);
  dim3 grid(cdiv(p.nout, kFrontTile), p.S);
  EnsureDynSmem(k_front<F>, smem);
  k_front<F><<<grid, kFrontTile, smem, st>>>(p);
}

void launch_front(const FrontParams& p, IqFormat fmt, cudaStream_t st)
{
  if (p.nout == 0 || p.S == 0)
    return;
  // u8 / s8: two bytes per sample; the tiled kernel's byte staging needs an even row base
  const bool bytes = fmt == kIqU8 || fmt == kIqS8;
  const bool tiled = p.order == 8 * p.ds && (p.ds == 1 || p.ds == 4 || p.ds == 5 || p.ds == 11) && p.coeff_host &&
                     (!bytes || ((reinterpret_cast<uintptr_t>(p.in) | (p.in_stride * 2)) & 1u) == 0);
  if (tiled)
  {
    FrontCoef cf;
    memset(&cf, 0, sizeof(cf));
    memcpy(cf.c, p.coeff_host, (p.order + 2) * sizeof(float));
    // TMA form: u8 / s8 rows that a tensor map can describe (16-byte aligned base and row pitch, whole 8-byte elements)
    if (bytes && p.tuner && (p.ds == 1 || p.ds == 5 || p.ds == 11) && p.n % 4 == 0 && p.n >= 4 &&
        (reinterpret_cast<uintptr_t>(p.in) & 15u) == 0 && (p.in_stride * 2) % 16 == 0)
    {
      if (fmt == kIqU8 ? launch_front_tma_ds<kIqU8>(p, cf, st) : launch_front_tma_ds<kIqS8>(p, cf, st))
        return;
    }
    switch (fmt)
    {
      case kIqU8: launch_front_tiled_ds<kIqU8>(p, cf, st); break;
      case kIqS8: launch_front_tiled_ds<kIqS8>(p, cf, st); break;
      case kIqS16: launch_front_tiled_ds<kIqS16>(p, cf, st); break;
      default: launch_front_tiled_ds<kIqCF32>(p, cf, st); break;
    }
    return;
  }
  switch (fmt)
  {
    case kIqU8: launch_front_generic<kIqU8>(p, st); break;
    case kIqS8: launch_front_generic<kIqS8>(p, st); break;
    case kIqS16: launch_front_generic<kIqS16>(p, st); break;
    default: launch_front_generic<kIqCF32>(p, st); break;
  }
}

void launch_front_tail(const FrontParams& p, IqFormat fmt, cudaStream_t st)
{
  if (p.S == 0 || p.n == 0)
    return;
  const size_t smem = (size_t)p.order * sizeof(float2);
  switch (fmt)
  {
    case kIqU8: k_front_tail<kIqU8><<<p.S, 256, smem, st>>>(p); break;
    case kIqS8: k_front_tail<kIqS8><<<p.S, 256, smem, st>>>(p); break;
    case kIqS16: k_front_tail<kIqS16><<<p.S, 256, smem, st>>>(p); break;
    default: k_front_tail<kIqCF32><<<p.S, 256, smem, st>>>(p); break;
  }
}

// ==================================================================================================
// lane kernels: one lane per stream, sequential in time (nonlinear recurrences).  Common plumbing:
// a warp owns 32 streams and walks the block in tiles of 32 samples; tiles move between HBM and shared memory
// with coalesced row accesses (cp.async for the next tile while the current one is computed) and are read /
// written by the lanes column-wise ([row][33] pitch: conflict-free).
// ==================================================================================================
constexpr unsigned kLT = 32;

__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem)
{
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* smem, const void* gmem)
{
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// rows s0 .. s0+31 of a [S][stride] array, columns t0 .. t0+31 -> dst[row][col]
__device__ __forceinline__ void tile_load_async(float (*dst)[kLT + 1], const float* base, size_t stride, unsigned s0,
                                                unsigned S, unsigned t0, unsigned n, unsigned lane)
{
  if (t0 + lane < n)
  {
    const unsigned rows = min(32u, S - s0);
    const float* g = base + (size_t)s0 * stride + t0 + lane;
    for (unsigned r = 0; r < rows; ++r, g += stride)
      cp_async_4(&dst[r][lane], g);
  }
}
__device__ __forceinline__ void tile_load_async(float2 (*dst)[kLT + 1], const float2* base, size_t stride, unsigned s0,
                                                unsigned S, unsigned t0, unsigned n, unsigned lane)
{
  if (t0 + lane < n)
  {
    const unsigned rows = min(32u, S - s0);
    const float2* g = base + (size_t)s0 * stride + t0 + lane;
    for (unsigned r = 0; r < rows; ++r, g += stride)
      cp_async_8(&dst[r][lane], g);
  }
}
template <typename T>
__device__ __forceinline__ void tile_store(T* base, size_t stride, unsigned s0, unsigned S, unsigned t0, unsigned n,
                                           unsigned lane, const T (*src)[kLT + 1])
{
  if (t0 + lane < n)
  {
    const unsigned rows = min(32u, S - s0);
    T* g = base + (size_t)s0 * stride + t0 + lane;
    for (unsigned r = 0; r < rows; ++r, g += stride)
      *g = src[r][lane];
  }
}

// named barriers (producer / consumer hand-off between the two warps of k_bb_lanes)
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// the same with the barrier id as an immediate: with register ids ptxas reserves all 16 named barriers for the CTA
// (EIATTR_NUM_BARRIERS = 16), and four such CTAs exhaust an SM's barriers (DESIGN.md section 10)
template <int ID>
__device__ __forceinline__ void bar_sync_imm() { asm volatile("bar.sync %0, 64;" ::"n"(ID) : "memory"); }
template <int ID>
__device__ __forceinline__ void bar_arrive_imm() { asm volatile("bar.arrive %0, 64;" ::"n"(ID) : "memory"); }

// --------------------------------------------------------------------------------------------------
// IF level meter: RMSLevelApprox over the first ceil(n/64) tuned samples, FmDecode.cpp:427,505-519
// --------------------------------------------------------------------------------------------------
template <int F>
__global__ void __launch_bounds__(128) k_if_level(FrontParams f, float* state)
{
  // one warp per stream: the |x|^2 terms are formed in parallel (coalesced), the float sum itself runs in sample
  // order on lane 0 (the reference's summation order, FmDecode.cpp:505-519)
  __shared__ float terms[4][1025];
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const unsigned s = blockIdx.x * 4 + warp;
  if (s >= f.S)
    return;
  const unsigned cnt = (f.n + 63) / 64;
  const size_t esz = IqBytes(F);
  const unsigned char* row = reinterpret_cast<const unsigned char*>(f.in) + (size_t)s * f.in_stride * esz;
  const float2* tuner = reinterpret_cast<const float2*>(f.tuner);
  float level = 0.0f;
  for (unsigned i0 = 0; i0 < cnt; i0 += 1024)
  {
    const unsigned m = min(1024u, cnt - i0);
    for (unsigned i = lane; i < m; i += 32)
    {
      const float2 t = tuned_sample<F>(row, i0 + i, f.idx0, f.lut, tuner);
      terms[warp][i] = addf(mulf(t.x, t.x), mulf(t.y, t.y));
    }
    __syncwarp();
    if (lane == 0)
      for (unsigned i = 0; i < m; ++i)
        level = addf(level, terms[warp][i]);
    __syncwarp();
  }
  if (lane == 0)
  {
    const float rms = sqrtf_rn(divf(level, (float)cnt));
    float* lv = state + (size_t)SF_IF_LEVEL * f.S + s;
    *lv = addf(mulf(0.95f, *lv), mulf(0.05f, rms));
  }
}

void launch_if_level(const FrontParams& p, float* state, IqFormat fmt, cudaStream_t st)
{
  if (p.S == 0 || p.n == 0)
    return;
  switch (fmt)
  {
    case kIqU8: k_if_level<kIqU8><<<cdiv(p.S, 4), 128, 0, st>>>(p, state); break;
    case kIqS8: k_if_level<kIqS8><<<cdiv(p.S, 4), 128, 0, st>>>(p, state); break;
    case kIqS16: k_if_level<kIqS16><<<cdiv(p.S, 4), 128, 0, st>>>(p, state); break;
    default: k_if_level<kIqCF32><<<cdiv(p.S, 4), 128, 0, st>>>(p, state); break;
  }
}

// --------------------------------------------------------------------------------------------------
// baseband lanes: warp 0 = FM-demodulator PLL (FmDecode.cpp:361-409), warp 1 = DC tracker + output scaling
// (:410-412), baseband meters (:439-442), 19 kHz pilot PLL (:143-229) and the 38 kHz demux multiply (:455-456).
// The two recurrences of a stream are independent except that the pilot PLL consumes the demodulator's output,
// so they run as a two-stage pipeline on two warps (two SM sub-partitions): a tile of NCO increments goes
// through a 2-slot shared-memory ring guarded by named barriers.  Per-sample cost is max(demod, pilot)
// instead of the sum.
// --------------------------------------------------------------------------------------------------
// --------------------------------------------------------------------------------------------------
// FM-demodulator PLL (FmDecode.cpp:361-409), time-parallel and still bit-exact.
// The loop is a fast contraction: two copies driven by the same input but started from different states
// (phase, increment) differ by a factor ~0.58 per sample (poles of the linearised loop), so after a short warm-up
// they coincide to the last bit.  k_demod_spec cuts the block into chunks of kDemodChunk samples and runs every
// (stream, chunk) on its own lane: chunk 0 starts from the carried state, chunk c > 0 starts `warm` samples
// early from a guess (phase 0, carried increment); the warm-up length is chosen by the host from the baseband rate (96 or 160
// samples: it only changes how often the repair pass has work).  It records the state it had at the chunk start and at the
// chunk end.  k_demod_fix then walks the chunks of a stream in order: where the recorded start state of chunk c is
// bit-identical to the (now known exact) end state of chunk c-1 the speculative outputs ARE the sequential ones;
// anywhere else -- in practice never on a tuned station, routinely on pure noise -- the chunk is recomputed
// sequentially from the exact state.  The result is always exactly the reference's sequential recurrence.
// --------------------------------------------------------------------------------------------------
#ifndef RFM_DEMOD_CHUNK
#define RFM_DEMOD_CHUNK 384
#endif
constexpr unsigned kDemodChunk = RFM_DEMOD_CHUNK; // multiples of the 32-sample tile

__global__ void __launch_bounds__(32) k_demod_spec(DemodSpecParams p)
{
  // Single-buffered tiles (12.6 KB per warp-CTA): ~17 warps per SM hide the tile-load latency of each other, which
  // is worth more here than overlapping a warp's own loads (the kernel is issue-bound once enough warps are resident).
  __shared__ float2 zin[32][kLT + 1];
  __shared__ float wout[32][kLT + 1];
  const unsigned lane = threadIdx.x;
  const unsigned s0 = blockIdx.x * 32;
  const unsigned s = s0 + lane;
  const unsigned c = blockIdx.y;
  const bool valid = s < p.S;
  const unsigned S = p.S;
  const unsigned t_begin = c * kDemodChunk;
  const unsigned t_end = min(p.nb, t_begin + kDemodChunk);
  const unsigned t_start = (c == 0) ? 0u : t_begin - p.warm; // p.warm <= kDemodChunk, multiple of the tile

  DemodState dm = {0.f, 0.f};
  if (valid)
  {
    dm.incr = p.state[SF_DEMOD_INCR * S + s];
    if (c == 0)
      dm.phase = p.state[SF_DEMOD_PHASE * S + s];
  }
  const float2* z = reinterpret_cast<const float2*>(p.z);
  const unsigned ntiles = (t_end - t_start + kLT - 1) / kLT;
  for (unsigned t = 0; t < ntiles; ++t)
  {
    const unsigned t0 = t_start + t * kLT;
    const unsigned tn = min(kLT, t_end - t0);
    tile_load_async(zin, z, p.z_stride, s0, S, t0, t_end, lane);
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp();
    if (t0 == t_begin && valid)
      p.st_start[(size_t)c * S + s] = make_float2(dm.phase, dm.incr);
    const DemodState tile_start = dm;
    bool bad = false;
    if (valid)
    {
      for (unsigned k = 0; k < tn; ++k)
      {
        const float2 x = zin[lane][k];
        demod_step_fast(dm, x.x, x.y, p.demod, bad);
        wout[lane][k] = dm.incr;
      }
    }
    if (__any_sync(0xffffffffu, bad))
    {
      dm = tile_start;
      if (valid)
      {
        for (unsigned k = 0; k < tn; ++k)
        {
          const float2 x = zin[lane][k];
          demod_step(dm, x.x, x.y, p.demod);
          wout[lane][k] = dm.incr;
        }
      }
    }
    __syncwarp();
    if (t0 >= t_begin)
      tile_store(p.incr, p.w_stride, s0, S, t0, t_end, lane, wout);
    __syncwarp();
  }
  if (valid)
    p.st_end[(size_t)c * S + s] = make_float2(dm.phase, dm.incr);
}

// Parallel repair pass: every (stream, chunk >= 1) whose assumed start state is not the end state of the previous
// chunk is recomputed from that end state -- all such chunks at once, one lane each.  A repaired chunk nearly
// always ends in the state it ended in before (the loop had converged inside the chunk), so one or two passes
// leave nothing for the sequential k_demod_fix, which remains as the unconditional guarantee.
__global__ void __launch_bounds__(32) k_demod_repair(DemodSpecParams p)
{
  __shared__ float2 zin[2][32][kLT + 1];
  __shared__ float wout[32][kLT + 1];
  const unsigned lane = threadIdx.x;
  const unsigned s0 = blockIdx.x * 32;
  const unsigned s = s0 + lane;
  const unsigned c = blockIdx.y + 1;
  const unsigned S = p.S;
  const bool valid = s < S;
  float2 prev_end = make_float2(0.f, 0.f), assumed = prev_end;
  if (valid)
  {
    prev_end = p.st_end[(size_t)(c - 1) * S + s];
    assumed = p.st_start[(size_t)c * S + s];
  }
  const bool mism = valid && (__float_as_uint(assumed.x) != __float_as_uint(prev_end.x) ||
                              __float_as_uint(assumed.y) != __float_as_uint(prev_end.y));
  const unsigned rows = __ballot_sync(0xffffffffu, mism);
  if (rows == 0u)
    return;
  if (mism && p.repairs)
    atomicAdd(p.repairs, 1ull);
  const unsigned t_begin = c * kDemodChunk;
  const unsigned t_end = min(p.nb, t_begin + kDemodChunk);
  DemodState dm = {prev_end.x, prev_end.y};
  const float2* z = reinterpret_cast<const float2*>(p.z);
  const unsigned ntiles = (t_end - t_begin + kLT - 1) / kLT;
  tile_load_async(zin[0], z, p.z_stride, s0, S, t_begin, t_end, lane);
  cp_async_commit();
  for (unsigned t = 0; t < ntiles; ++t)
  {
    const unsigned b = t & 1u, t0 = t_begin + t * kLT;
    const unsigned tn = min(kLT, t_end - t0);
    if (t + 1 < ntiles)
      tile_load_async(zin[b ^ 1u], z, p.z_stride, s0, S, t0 + kLT, t_end, lane);
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    const DemodState tile_start = dm;
    bool bad = false;
    if (mism)
    {
      for (unsigned k = 0; k < tn; ++k)
      {
        const float2 x = zin[b][lane][k];
        demod_step_fast(dm, x.x, x.y, p.demod, bad);
        wout[lane][k] = dm.incr;
      }
    }
    if (__any_sync(0xffffffffu, bad))
    {
      dm = tile_start;
      if (mism)
      {
        for (unsigned k = 0; k < tn; ++k)
        {
          const float2 x = zin[b][lane][k];
          demod_step(dm, x.x, x.y, p.demod);
          wout[lane][k] = dm.incr;
        }
      }
    }
    __syncwarp();
    // only the repaired rows are written back
    if (t0 + lane < t_end)
      for (unsigned r = 0; r < 32; ++r)
        if ((rows >> r) & 1u)
          p.incr[(size_t)(s0 + r) * p.w_stride + t0 + lane] = wout[r][lane];
    __syncwarp();
  }
  if (mism)
  {
    p.st_start[(size_t)c * S + s] = prev_end;
    p.st_end[(size_t)c * S + s] = make_float2(dm.phase, dm.incr);
  }
}

__global__ void __launch_bounds__(32) k_demod_fix(DemodSpecParams p)
{
  const unsigned s = blockIdx.x * 32 + threadIdx.x;
  const bool valid = s < p.S;
  const unsigned S = p.S;
  const unsigned nchunks = (p.nb + kDemodChunk - 1) / kDemodChunk;
  float2 cur = make_float2(0.f, 0.f);
  if (valid)
    cur = p.st_end[s];
  const float2* z = reinterpret_cast<const float2*>(p.z) + (size_t)s * p.z_stride;
  float* w = p.incr + (size_t)s * p.w_stride;
  for (unsigned c = 1; c < nchunks; ++c)
  {
    float2 assumed = cur, end = cur;
    if (valid)
    {
      assumed = p.st_start[(size_t)c * S + s];
      end = p.st_end[(size_t)c * S + s];
    }
    const bool mism = valid && (__float_as_uint(assumed.x) != __float_as_uint(cur.x) ||
                                __float_as_uint(assumed.y) != __float_as_uint(cur.y));
    if (__any_sync(0xffffffffu, mism))
    {
      if (mism)
      {
        if (p.repairs)
          atomicAdd(p.repairs, 1ull);
        // the speculation missed for this stream: redo the chunk from the exact state (rare; direct global access)
        DemodState dm = {cur.x, cur.y};
        const unsigned t1 = min(p.nb, (c + 1) * kDemodChunk);
        for (unsigned t = c * kDemodChunk; t < t1; ++t)
        {
          const float2 x = z[t];
          demod_step(dm, x.x, x.y, p.demod);
          w[t] = dm.incr;
        }
        end = make_float2(dm.phase, dm.incr);
      }
    }
    cur = end;
  }
  if (valid)
  {
    p.state[SF_DEMOD_PHASE * S + s] = cur.x;
    p.state[SF_DEMOD_INCR * S + s] = cur.y;
  }
}

void launch_demod_spec(const DemodSpecParams& p, cudaStream_t st)
{
  if (p.S == 0 || p.nb == 0)
    return;
  const unsigned nchunks = cdiv(p.nb, kDemodChunk);
  dim3 grid(cdiv(p.S, 32), nchunks);
  k_demod_spec<<<grid, 32, 0, st>>>(p);
}

void launch_demod_fix(const DemodSpecParams& p, cudaStream_t st)
{
  if (p.S == 0 || p.nb == 0)
    return;
  const unsigned nchunks = cdiv(p.nb, kDemodChunk);
  if (nchunks > 1)
  {
    dim3 grid(cdiv(p.S, 32), nchunks - 1);
    k_demod_repair<<<grid, 32, 0, st>>>(p);
  }
  k_demod_fix<<<cdiv(p.S, 32), 32, 0, st>>>(p);
}

unsigned demod_chunks(unsigned nb) { return cdiv(nb, kDemodChunk); }

// --------------------------------------------------------------------------------------------------
// baseband lanes: warp 0 = DC tracker + output scaling (FmDecode.cpp:410-412) and baseband meters (:439-442);
// warp 1 = 19 kHz pilot PLL (:143-229) and the 38 kHz demux multiply (:455-456).  Both are one-lane-per-stream
// recurrences; the pilot PLL consumes the baseband the first warp produces, so they run as a two-stage pipeline on
// two warps (two SM sub-partitions): tiles of baseband go through a 2-slot shared-memory ring guarded by named
// barriers, and the pilot warp -- the long pole of the whole chain -- carries nothing but its own recurrence.
// --------------------------------------------------------------------------------------------------
struct LanesSmem
{
  float win[2][32][kLT + 1];   // NCO increments from the demodulator
  float ring[2][32][kLT + 1];  // baseband, warp 0 -> warp 1
  float rawt[32][kLT + 1];
  double kd[13];               // sincos constants / pilot constants, re-read ONCE per block with volatile loads
  float kf[8];
};

// FAKE_SINCOS: RFM_DEBUG_FAKE_SINCOS timing experiment (wrong results, experiments build only).  IMMBAR: barrier ids as
// immediates (5 named barriers per CTA instead of the 16 ptxas reserves for register ids, so up to 12 CTAs fit on an
// SM; same hand-off) -- the product form; the register-id form remains as an experiment (RFM_LANES_REGBAR).
template <bool FAKE_SINCOS, bool IMMBAR = false, bool SPEC = false, bool XUFREE = false>
__global__ void __launch_bounds__(64) k_bb_lanes(LanesParams p)
{
  __shared__ LanesSmem sm;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned role = (threadIdx.x >> 5) ^ (p.role_swap & blockIdx.x & 1u);
  const unsigned s0 = blockIdx.x * 32;
  const unsigned s = s0 + lane;
  const bool valid = s < p.S;
  const unsigned S = p.S;
  float* st = p.state;
  const unsigned ntiles = (p.nb + kLT - 1) / kLT;
  enum { BAR_FULL = 1, BAR_EMPTY = 3 };
  auto sync_bar = [](int base, unsigned b) {
    if (!IMMBAR)
      bar_sync(base + (int)b, 64);
    else if (base == BAR_FULL)
    {
      if (b) bar_sync_imm<BAR_FULL + 1>(); else bar_sync_imm<BAR_FULL>();
    }
    else
    {
      if (b) bar_sync_imm<BAR_EMPTY + 1>(); else bar_sync_imm<BAR_EMPTY>();
    }
  };
  auto arrive_bar = [](int base, unsigned b) {
    if (!IMMBAR)
      bar_arrive(base + (int)b, 64);
    else if (base == BAR_FULL)
    {
      if (b) bar_arrive_imm<BAR_FULL + 1>(); else bar_arrive_imm<BAR_FULL>();
    }
    else
    {
      if (b) bar_arrive_imm<BAR_EMPTY + 1>(); else bar_arrive_imm<BAR_EMPTY>();
    }
  };

  if (role == 0)
  {
    // ---------------- producer: DC tracker, output scaling, meters ----------------
    float dc = 0.0f, vsum = 0.0f, vsumsq = 0.0f;
    if (valid)
      dc = st[SF_DEMOD_DC * S + s];
    tile_load_async(sm.win[0], p.incr, p.w_stride, s0, S, 0, p.nb, lane);
    cp_async_commit();
    for (unsigned t = 0; t < ntiles; ++t)
    {
      const unsigned b = t & 1u, t0 = t * kLT;
      const unsigned tn = min(kLT, p.nb - t0);
      if (t + 1 < ntiles)
        tile_load_async(sm.win[b ^ 1u], p.incr, p.w_stride, s0, S, t0 + kLT, p.nb, lane);
      cp_async_commit();
      cp_async_wait<1>();
      __syncwarp();
      if (t >= 2)
        sync_bar(BAR_EMPTY, b);
      if (XUFREE)
      {
        // conversions on the integer pipe (rfm_math.cuh); a flagged tile is replayed with the conversion instructions
        const float dc0 = dc, vs0 = vsum, vq0 = vsumsq;
        bool bad = false;
        if (valid)
        {
          for (unsigned k = 0; k < tn; ++k)
          {
            const float bb = demod_output_bits(sm.win[b][lane][k], dc, p.demod.gain, bad);
            vsum = addf(vsum, bb);
            vsumsq = addf(vsumsq, mulf(bb, bb));
            sm.ring[b][lane][k] = bb;
          }
        }
        if (__any_sync(0xffffffffu, bad))
        {
          dc = dc0; vsum = vs0; vsumsq = vq0;
          if (valid)
          {
            for (unsigned k = 0; k < tn; ++k)
            {
              const float bb = demod_output(sm.win[b][lane][k], dc, p.demod.gain);
              vsum = addf(vsum, bb);
              vsumsq = addf(vsumsq, mulf(bb, bb));
              sm.ring[b][lane][k] = bb;
            }
          }
        }
      }
      else if (valid)
      {
        for (unsigned k = 0; k < tn; ++k)
        {
          const float bb = demod_output(sm.win[b][lane][k], dc, p.demod.gain);
          vsum = addf(vsum, bb);                       // SamplesMeanRMS, FmDecode.cpp:522-539
          vsumsq = addf(vsumsq, mulf(bb, bb));
          sm.ring[b][lane][k] = bb;
        }
      }
      __threadfence_block();
      arrive_bar(BAR_FULL, b);
      __syncwarp();
      tile_store(p.bbV + p.a_hist, p.a_stride, s0, S, t0, p.nb, lane, sm.ring[b]);
      __syncwarp();
    }
    if (valid)
    {
      st[SF_DEMOD_DC * S + s] = dc;
      // baseband meters, FmDecode.cpp:439-442
      const float mean = divf(vsum, (float)p.nb);
      const float rms = sqrtf_rn(divf(vsumsq, (float)p.nb));
      st[SF_BB_MEAN * S + s] = addf(mulf(0.95f, st[SF_BB_MEAN * S + s]), mulf(0.05f, mean));
      st[SF_BB_LEVEL * S + s] = addf(mulf(0.95f, st[SF_BB_LEVEL * S + s]), mulf(0.05f, rms));
    }
  }
  else
  {
    // ---------------- consumer: pilot PLL, demux multiply ----------------
    PilotState pl = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1000.0f};
    // loop constants through shared memory and volatile loads: held in registers for the whole block (rfm_math.cuh)
    if (lane < 13)
      sm.kd[lane] = kSinCosDev[lane];
    if (lane == 0)
    {
      sm.kf[0] = p.pilot.minfreq; sm.kf[1] = p.pilot.maxfreq; sm.kf[2] = p.pilot.b0; sm.kf[3] = p.pilot.a1;
      sm.kf[4] = p.pilot.a2; sm.kf[5] = p.pilot.lb0; sm.kf[6] = p.pilot.lb1;
    }
    __syncwarp();
    SinCosRegs sca;
#pragma unroll
    for (int i = 0; i < 13; ++i)
      sca.k[i] = *reinterpret_cast<volatile double*>(&sm.kd[i]);
    PilotConstDev pk = p.pilot;
    {
      volatile float* kf = sm.kf;
      pk.minfreq = kf[0]; pk.maxfreq = kf[1]; pk.b0 = kf[2]; pk.a1 = kf[3]; pk.a2 = kf[4]; pk.lb0 = kf[5]; pk.lb1 = kf[6];
    }
    if (valid)
    {
      pl.phase = st[SF_PILOT_PHASE * S + s];
      pl.freq = st[SF_PILOT_FREQ * S + s];
      pl.i1 = st[SF_PILOT_I1 * S + s];
      pl.i2 = st[SF_PILOT_I2 * S + s];
      pl.q1 = st[SF_PILOT_Q1 * S + s];
      pl.q2 = st[SF_PILOT_Q2 * S + s];
      pl.x1 = st[SF_PILOT_X1 * S + s];
      pl.level = 1000.0f; // FmDecode.cpp:147
    }
    // (ps, pc) = sincos(phase) carried from sample to sample by the speculative form (rfm_math.cuh: rfm_sincos_predict)
    PilotCarry sc = {0.0f, 1.0f};
    if (SPEC)
      rfm_sincos(pl.phase, &sc.ps, &sc.pc);
    unsigned backoff = 0; // tiles left in the plain form after the speculation was refused (unlocked loop, noise)
    for (unsigned t = 0; t < ntiles; ++t)
    {
      const unsigned b = t & 1u, t0 = t * kLT;
      const unsigned tn = min(kLT, p.nb - t0);
      sync_bar(BAR_FULL, b);
      // branch-free fast paths; if any lane raised the sticky flag the tile is replayed with the next safer form:
      // speculative sincos -> direct branch-free sincos -> the exact routines.  All three produce pilot_step's bits.
      const PilotState pl_start = pl;
      bool bad = false;
      bool done = false;
      if (SPEC && backoff == 0)
      {
        if (valid)
        {
#pragma unroll 2
          for (unsigned k = 0; k < tn; ++k)
          {
            const float bb = sm.ring[b][lane][k];
            const float p38 = pilot_step_spec(pl, sc, bb, pk, sca, bad);
            sm.rawt[lane][k] = mulf(p38, mulf(2.0f, bb)); // FmDecode.cpp:455-456
          }
        }
        done = !__any_sync(0xffffffffu, bad);
        if (!done)
        {
          pl = pl_start;
          bad = false;
          backoff = 8;
        }
      }
      else if (SPEC)
        --backoff;
      if (!done)
      {
        if (valid)
        {
#pragma unroll 2
          for (unsigned k = 0; k < tn; ++k)
          {
            const float bb = sm.ring[b][lane][k];
            const float p38 = pilot_step_fast<FAKE_SINCOS, XUFREE>(pl, bb, pk, sca, bad);
            sm.rawt[lane][k] = mulf(p38, mulf(2.0f, bb)); // FmDecode.cpp:455-456
          }
        }
        if (__any_sync(0xffffffffu, bad))
        {
          pl = pl_start;
          if (valid)
          {
            for (unsigned k = 0; k < tn; ++k)
            {
              const float bb = sm.ring[b][lane][k];
              const float p38 = pilot_step(pl, bb, p.pilot);
              sm.rawt[lane][k] = mulf(p38, mulf(2.0f, bb));
            }
          }
        }
        if (SPEC && backoff == 0)
          rfm_sincos(pl.phase, &sc.ps, &sc.pc); // the next tile speculates again
      }
      if (t + 2 < ntiles)
        arrive_bar(BAR_EMPTY, b);
      __syncwarp();
      tile_store(p.rawV + p.a_hist, p.a_stride, s0, S, t0, p.nb, lane, sm.rawt);
      __syncwarp();
    }
    if (valid)
    {
      st[SF_PILOT_PHASE * S + s] = pl.phase;
      st[SF_PILOT_FREQ * S + s] = pl.freq;
      st[SF_PILOT_I1 * S + s] = pl.i1;
      st[SF_PILOT_I2 * S + s] = pl.i2;
      st[SF_PILOT_Q1 * S + s] = pl.q1;
      st[SF_PILOT_Q2 * S + s] = pl.q2;
      st[SF_PILOT_X1 * S + s] = pl.x1;
      st[SF_PILOT_LEVEL * S + s] = pl.level;
      // lock detector, FmDecode.cpp:219-228
      int lock_cnt = __float_as_int(st[SF_PILOT_LOCKCNT * S + s]);
      if (mulf(2.0f, pl.level) > p.pilot.minsignal)
      {
        if (lock_cnt < p.pilot.lock_delay)
          lock_cnt += (int)p.nb;
      }
      else
        lock_cnt = 0;
      st[SF_PILOT_LOCKCNT * S + s] = __int_as_float(lock_cnt);
      st[(SF_STEREO + p.parity) * S + s] = __int_as_float(lock_cnt >= p.pilot.lock_delay ? 1 : 0);
    }
  }
}

void launch_bb_lanes(const LanesParams& p_in, cudaStream_t st)
{
  if (p_in.S == 0 || p_in.nb == 0)
    return;
  LanesParams p = p_in;
  p.role_swap = 0;
#ifdef RFM_EXPERIMENTS
  static const unsigned swap = (unsigned)KnobInt(RFM_KNOB("RFM_LANES_SWAP"), 0) & 1u;
  p.role_swap = swap;
  // experiment (with RFM_LANES_SMS): ask for the largest shared-memory carve-out so that 8 lanes CTAs fit on one SM
  static const bool carve = KnobInt(RFM_KNOB("RFM_LANES_CARVEOUT"), 0) != 0;
  if (carve)
  {
    static bool done[64] = {false};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !done[dev])
    {
      cudaFuncSetAttribute(k_bb_lanes<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      done[dev] = true;
    }
  }
  // measurement aid: reserve extra (unused) dynamic shared memory so fewer throughput CTAs share the lanes' SMs
  static const int reserve_kb = KnobInt(RFM_KNOB("RFM_LANES_RESERVE_KB"), 0);
  static const bool fake = KnobInt(RFM_KNOB("RFM_DEBUG_FAKE_SINCOS"), 0) != 0;
  if (reserve_kb > 0)
  {
    EnsureDynSmem(k_bb_lanes<false, true>, (size_t)reserve_kb * 1024);
    EnsureDynSmem(k_bb_lanes<true, true>, (size_t)reserve_kb * 1024);
  }
  static const bool fake_ = fake;
  (void)fake_;
  if (fake)
    return (void)k_bb_lanes<true, true><<<cdiv(p.S, 32), 64, (size_t)reserve_kb * 1024, st>>>(p);
  if (reserve_kb > 0)
    return (void)k_bb_lanes<false, true><<<cdiv(p.S, 32), 64, (size_t)reserve_kb * 1024, st>>>(p);
  // speculative sincos (pilot_step_spec): bit-exact (tests/test_host_steps.py, 2e9-case fuzz) but measured slower:
  // 139 instructions per sample against 94, 1.06 ms alone against 0.96, 2.34 ms under load against 2.06 (DESIGN.md 10)
  static const bool spec = KnobInt(RFM_KNOB("RFM_LANES_SPEC"), 0) != 0;
  if (spec)
    return (void)k_bb_lanes<false, true, true><<<cdiv(p.S, 32), 64, 0, st>>>(p);
  static const int xufree = KnobInt(RFM_KNOB("RFM_LANES_XUFREE"), 0);
  if (xufree == 1)
    return p.packed ? (void)k_bb_lanes<false, true, false, true><<<cdiv(p.S, 32), 64, 0, st>>>(p)
                    : (void)k_bb_lanes<false, false, false, true><<<cdiv(p.S, 32), 64, 0, st>>>(p);
  static const int immbar = KnobInt(RFM_KNOB("RFM_LANES_IMMBAR"), -1);
  if (immbar == 1)
    return (void)k_bb_lanes<false, true><<<cdiv(p.S, 32), 64, 0, st>>>(p);
  if (immbar == 0)
    return (void)k_bb_lanes<false, false><<<cdiv(p.S, 32), 64, 0, st>>>(p);
#endif
  // Barrier ids as immediates let up to 12 lanes CTAs share an SM, which is what an SM partition of a few SMs needs;
  // without a partition that packing is harmful (co-resident pilot warps queue for the SM's one conversion / MUFU
  // pipe: 2.28 ms per step against 2.08), and the register-id form's 16 reserved barriers keep it at 4 CTAs per SM.
  // (The conversions of the pilot / DC-tracker steps on the integer pipe -- rfm_f2d_bits / rfm_d2f_bits, bit-exact --
  // were measured too, RFM_LANES_XUFREE=1 in the experiments build: 130 + 57 instructions per sample instead of
  // 94 + 16 trade the XU queue for the half-rate ALU pipe and lose: 1.83 ms on 24 SMs against 1.44.)
  if (p.packed)
    k_bb_lanes<false, true><<<cdiv(p.S, 32), 64, 0, st>>>(p);
  else
    k_bb_lanes<false, false><<<cdiv(p.S, 32), 64, 0, st>>>(p);
}


// ==================================================================================================
// fractional resampler (mono + stereo), DownConvert.cpp:195-233
// ==================================================================================================
constexpr unsigned kResTile = 64;

__device__ __forceinline__ float res_pos(float p0, float pstep, unsigned i)
{
  return addf(p0, mulf((float)i, pstep)); // pf = p + i * pstep, DownConvert.cpp:224
}

__global__ void __launch_bounds__(kResTile) k_resample(ResampleParams p, unsigned max_span)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* s_coef = reinterpret_cast<float*>(smem_raw);
  float* Xm = s_coef + p.order + 2;
  float* Xs = Xm + max_span;

  const unsigned tid = threadIdx.x;
  const unsigned s = blockIdx.y;
  const unsigned i0 = blockIdx.x * kResTile;
  const unsigned i1 = min(i0 + kResTile, p.na) - 1;

  for (unsigned i = tid; i < p.order + 2; i += kResTile)
    s_coef[i] = p.coeff[i];

  const unsigned lo = (unsigned)__float2int_rz(res_pos(p.pos_frac, p.pstep, i0));
  const unsigned hi = (unsigned)__float2int_rz(res_pos(p.pos_frac, p.pstep, i1)) + p.order;
  const unsigned span = hi - lo + 1;
  const float* bb = p.bbV + (size_t)s * p.a_stride;
  const float* raw = p.rawV + (size_t)s * p.a_stride;
  for (unsigned v = tid; v < span; v += kResTile)
  {
    Xm[v] = bb[lo + v];
    Xs[v] = raw[lo + v];
  }
  __syncthreads();

  const unsigned i = i0 + tid;
  if (i <= i1)
  {
    const float pf = res_pos(p.pos_frac, p.pstep, i);
    const unsigned pi = (unsigned)__float2int_rz(pf);
    const float k1 = subf(pf, (float)pi);
    const float k0 = subf(1.0f, k1);
    // y = sum_{j=0..order} (c[j] k0 + c[j+1] k1) * V[order + pi - j]
    const unsigned base = pi - lo + p.order;
    float ym = 0.0f, ys = 0.0f;
    float cj = s_coef[0];
    for (unsigned j = 0; j <= p.order; ++j)
    {
      const float cn = s_coef[j + 1];
      const float k = addf(mulf(cj, k0), mulf(cn, k1));
      ym = addf(ym, mulf(k, Xm[base - j]));
      ys = addf(ys, mulf(k, Xs[base - j]));
      cj = cn;
    }
    p.lpM[(size_t)s * p.lp_stride + p.lp_hist + i] = ym;
    p.lpS[(size_t)s * p.lp_stride + p.lp_hist + i] = ys;
  }
}

void launch_resample(const ResampleParams& p, cudaStream_t st)
{
  if (p.na == 0 || p.S == 0)
    return;
  const unsigned max_span = (unsigned)((float)kResTile * p.pstep) + p.order + 8;
  const size_t smem = (size_t)(p.order + 2 + 2 * max_span) * sizeof(float);
  EnsureDynSmem(k_resample, smem);
  dim3 grid(cdiv(p.na, kResTile), p.S);
  k_resample<<<grid, kResTile, smem, st>>>(p, max_span);
}

// --------------------------------------------------------------------------------------------------
// Tiled form.  The output positions pf = p + i * pstep and with them the interpolated taps
// k[i][j] = c[j] (1 - k1_i) + c[j+1] k1_i are the same for EVERY stream of the decoder (lock-step), so they are
// formed once per block by k_res_taps (DownConvert.cpp:203-224, same float operations) and shared:
//   * outputs are handled in groups of 4 consecutive ones; a group's taps are stored against a common time axis that
//     starts at a multiple of 4 samples and is a multiple of 4 long (zero outside an output's own window: adding +-0
//     leaves a running sum that started at +0 unchanged), 4 taps per time step as one float4;
//   * k_resample_tiled: lane = stream, warp = group.  The [32 streams][span] input tiles of both channels and the
//     groups' taps travel to shared memory with 16-byte cp.async copies (no registers, no per-element stores); rows
//     keep a 16-byte aligned pitch of 4 * odd floats, so a lane's LDS.128 of four consecutive samples is
//     conflict-free across the 8 lanes of a quarter warp.  A warp walks its group from the newest sample down --
//     every output receives its taps in ascending j, the reference's order (DownConvert.cpp:210-222) -- with
//     6 LDS.128 (4 tap vectors, 4 mono + 4 L-R samples) per 64 individually rounded multiply / add operations;
//   * the tile (GB groups) is sized so that two CTAs fit on an SM: one stages while the other computes.
// --------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_res_taps(ResTapsParams p)
{
  const unsigned g = blockIdx.x;
  __shared__ int s_pi[4];
  __shared__ float s_k0[4], s_k1[4];
  if (threadIdx.x < 4)
  {
    const unsigned i = 4 * g + threadIdx.x;
    const float pf = res_pos(p.pos_frac, p.pstep, i);
    const int pi = __float2int_rz(pf);
    const float k1 = subf(pf, (float)pi);
    s_pi[threadIdx.x] = (i < p.na) ? pi : -1;
    s_k1[threadIdx.x] = k1;
    s_k0[threadIdx.x] = subf(1.0f, k1);
  }
  __syncthreads();
  // valid outputs of this group: 0 .. cnt-1 (cnt >= 1)
  unsigned cnt = 0;
  for (unsigned r = 0; r < 4; ++r)
    cnt += s_pi[r] >= 0;
  const int vlo = s_pi[0] & ~3;                  // V index (history included) of the oldest sample of output 0, aligned down
  const int vhi = (int)p.order + s_pi[cnt - 1];  // newest sample of the last valid output
  const int L = (vhi - vlo + 1 + 3) & ~3;
  if (threadIdx.x == 0)
  {
    p.meta[2 * g] = vlo;
    p.meta[2 * g + 1] = L;
  }
  float4* kk = reinterpret_cast<float4*>(p.kk) + (size_t)g * p.lp;
  for (int tt = threadIdx.x; tt < (int)p.lp; tt += blockDim.x)
  {
    float v[4];
    for (unsigned r = 0; r < 4; ++r)
    {
      const int j = (int)p.order + s_pi[r] - (vlo + tt); // tap of output r that meets V = vlo + tt
      v[r] = 0.0f;
      if (s_pi[r] >= 0 && j >= 0 && j <= (int)p.order)
        v[r] = addf(mulf(p.coeff[j], s_k0[r]), mulf(p.coeff[j + 1], s_k1[r]));
    }
    kk[tt] = make_float4(v[0], v[1], v[2], v[3]);
  }
}

void launch_res_taps(const ResTapsParams& p, cudaStream_t st)
{
  if (p.na == 0)
    return;
  k_res_taps<<<cdiv(p.na, 4), 128, 0, st>>>(p);
}

__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem)
{
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}

template <int GB, bool FUSED> // groups of 4 outputs per CTA == warps per CTA
__global__ void __launch_bounds__(32 * GB) k_resample_tiled(ResampleParams p, unsigned pitch)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float4* KK = reinterpret_cast<float4*>(smem_raw);                 // [GB][lp]
  float* X = reinterpret_cast<float*>(KK + (size_t)GB * p.lp);      // [2][32][pitch]
  __shared__ int s_meta[2 * GB];

  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const unsigned ngroups = (p.na + 3) / 4;
  const unsigned g0 = blockIdx.x * GB;
  const unsigned gn = min((unsigned)GB, ngroups - g0);
  const unsigned s0 = blockIdx.y * 32;
  const unsigned rows = min(32u, p.S - s0);
  if (tid < 2 * gn)
    s_meta[tid] = p.meta[2 * g0 + tid];
  __syncthreads();
  const int v0 = s_meta[0];                                                  // multiple of 4
  const int nq = (s_meta[2 * (gn - 1)] + s_meta[2 * (gn - 1) + 1] - v0) >> 2; // 16-byte columns of the CTA's V range
  {
    const float4* ksrc = reinterpret_cast<const float4*>(p.kk) + (size_t)g0 * p.lp;
    for (unsigned i = tid; i < gn * p.lp; i += 32 * GB)
      cp_async_16(&KK[i], &ksrc[i]);
  }
  for (unsigned r = warp; r < rows; r += GB)
  {
    const float* b0 = p.bbV + (size_t)(s0 + r) * p.a_stride + v0;
    const float* b1 = p.rawV + (size_t)(s0 + r) * p.a_stride + v0;
    float* x0 = X + (size_t)r * pitch;
    float* x1 = X + (size_t)(32 + r) * pitch;
    for (int c = lane; c < nq; c += 32)
    {
      cp_async_16(x0 + 4 * c, b0 + 4 * c);
      cp_async_16(x1 + 4 * c, b1 + 4 * c);
    }
  }
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  if (lane >= rows || warp >= gn)
    return;
  const int off = s_meta[2 * warp] - v0;
  const int Lq = s_meta[2 * warp + 1] >> 2;
  const float4* kk = KK + (size_t)warp * p.lp;
  const float4* x0 = reinterpret_cast<const float4*>(X + (size_t)lane * pitch + off);
  const float4* x1 = reinterpret_cast<const float4*>(X + (size_t)(32 + lane) * pitch + off);
  float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
#define RS_STEP(k, m, sv)                                                                     \
  a[0] = macf<FUSED>(a[0], (k).x, m); a[1] = macf<FUSED>(a[1], (k).y, m);                     \
  a[2] = macf<FUSED>(a[2], (k).z, m); a[3] = macf<FUSED>(a[3], (k).w, m);                     \
  b[0] = macf<FUSED>(b[0], (k).x, sv); b[1] = macf<FUSED>(b[1], (k).y, sv);                   \
  b[2] = macf<FUSED>(b[2], (k).z, sv); b[3] = macf<FUSED>(b[3], (k).w, sv);
  // software pipeline: the six vectors of step q - 1 are in flight while step q is multiplied out (with three warps
  // per scheduler the shared-memory latency was this loop's main stall: 1.4 short-scoreboard cycles per issue)
  float4 m = x0[Lq - 1], sv = x1[Lq - 1];
  float4 k3 = kk[4 * Lq - 1], k2 = kk[4 * Lq - 2], k1 = kk[4 * Lq - 3], k0 = kk[4 * Lq - 4];
#pragma unroll 2
  for (int q = Lq - 1; q > 0; --q)
  {
    const float4 mn = x0[q - 1], svn = x1[q - 1];
    const float4 n3 = kk[4 * q - 1], n2 = kk[4 * q - 2], n1 = kk[4 * q - 3], n0 = kk[4 * q - 4];
    RS_STEP(k3, m.w, sv.w)
    RS_STEP(k2, m.z, sv.z)
    RS_STEP(k1, m.y, sv.y)
    RS_STEP(k0, m.x, sv.x)
    m = mn; sv = svn; k3 = n3; k2 = n2; k1 = n1; k0 = n0;
  }
  RS_STEP(k3, m.w, sv.w)
  RS_STEP(k2, m.z, sv.z)
  RS_STEP(k1, m.y, sv.y)
  RS_STEP(k0, m.x, sv.x)
#undef RS_STEP
  const unsigned i = 4 * (g0 + warp);
  const bool vec = i + 4 <= p.na && ((p.lp_hist | p.lp_stride) & 3u) == 0;
  float* oM = p.lpM + (size_t)(s0 + lane) * p.lp_stride + p.lp_hist + i;
  float* oS = p.lpS + (size_t)(s0 + lane) * p.lp_stride + p.lp_hist + i;
  if (vec)
  {
    *reinterpret_cast<float4*>(oM) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(oS) = make_float4(b[0], b[1], b[2], b[3]);
  }
  else
    for (unsigned r = 0; r < 4 && i + r < p.na; ++r)
    {
      oM[r] = a[r];
      oS[r] = b[r];
    }
}

template <int GB>
static void launch_resample_tiled_gb(const ResampleParams& p, unsigned pitch, size_t smem, cudaStream_t st)
{
  dim3 grid(cdiv((p.na + 3) / 4, GB), cdiv(p.S, 32));
  if (p.fused)
  {
    EnsureDynSmem(k_resample_tiled<GB, true>, smem);
    k_resample_tiled<GB, true><<<grid, 32 * GB, smem, st>>>(p, pitch);
  }
  else
  {
    EnsureDynSmem(k_resample_tiled<GB, false>, smem);
    k_resample_tiled<GB, false><<<grid, 32 * GB, smem, st>>>(p, pitch);
  }
}

void launch_resample_tiled(const ResampleParams& p, cudaStream_t st)
{
  if (p.na == 0 || p.S == 0)
    return;
  // rows must allow 16-byte copies from any multiple of 4 samples
  const bool aligned = ((reinterpret_cast<uintptr_t>(p.bbV) | reinterpret_cast<uintptr_t>(p.rawV)) & 15u) == 0 &&
                       (p.a_stride & 3u) == 0 && (p.lp & 3u) == 0;
  auto need = [&](unsigned gb, unsigned* pitch) {
    // V range of gb groups: 4 gb outputs apart + one window + the alignment slack at both ends
    const unsigned span_max = ((unsigned)(4.0f * gb * p.pstep) + p.order + 1 + 8 + 3) & ~3u;
    *pitch = span_max | 4u; // multiple of 4 with pitch / 4 odd: conflict-free LDS.128 across a quarter warp
    return (size_t)gb * p.lp * sizeof(float4) + (size_t)2 * 32 * *pitch * sizeof(float);
  };
  unsigned pitch = 0;
  size_t smem = 0;
  // the largest tile of which two CTAs fit on an SM (one stages while the other computes); else the largest that fits
  constexpr size_t kTwo = 113 * 1024, kOne = 220 * 1024;
#define RFM_RS(GBV, LIM)                                              \
  if (aligned && (smem = need(GBV, &pitch)) <= (LIM))                 \
    return launch_resample_tiled_gb<GBV>(p, pitch, smem, st);
  RFM_RS(8, kTwo) RFM_RS(6, kTwo) RFM_RS(4, kTwo) RFM_RS(3, kTwo) RFM_RS(2, kTwo)
  RFM_RS(8, kOne) RFM_RS(4, kOne) RFM_RS(2, kOne) RFM_RS(1, kOne)
#undef RFM_RS
  launch_resample(p, st); // very long filters: untiled form
}

// ==================================================================================================
// cFirFilter::Process / ProcessTwo, FirFilter.cpp:330-413
// y[g] = sum over j = 0..N-1 of h[k_j] x[g - k_j],  k_j = (g + j) mod N: the circular delay line is
// walked in buffer order, so the first tap of the sum rotates with the running sample count g.
// ==================================================================================================
constexpr unsigned kFirTile = 128;

constexpr unsigned kFirOut = 4 * kFirTile; // outputs per CTA (4 per thread, strided by the CTA width)

template <int MODE> // 0 real, 1 real pair, 2 complex
__global__ void __launch_bounds__(kFirTile) k_rotfir(RotFirParams p)
{
  // CTA = 512 consecutive outputs of one stream; the input window [taps - 1 | 512] is staged in shared memory
  __shared__ float s_coef[kMaxFirTapsDev];
  __shared__ float s_a[(MODE == 2 ? 2 : 1) * (kMaxFirTapsDev + kFirOut)];
  __shared__ float s_b[MODE == 1 ? (kMaxFirTapsDev + kFirOut) : 1];
  const unsigned tid = threadIdx.x;
  const unsigned N = p.taps;
  const unsigned s = blockIdx.y;
  const unsigned i0 = blockIdx.x * kFirOut;
  const unsigned nt = min(kFirOut, p.n - i0);
  for (unsigned i = tid; i < N; i += kFirTile)
    s_coef[i] = p.coef[i];
  const unsigned wlen = N - 1 + nt; // V indices i0 .. i0 + wlen - 1
  if (MODE == 2)
  {
    const float2* x = reinterpret_cast<const float2*>(p.inA) + (size_t)s * p.in_stride + i0;
    for (unsigned i = tid; i < wlen; i += kFirTile)
      reinterpret_cast<float2*>(s_a)[i] = x[i];
  }
  else
  {
    const float* xa = p.inA + (size_t)s * p.in_stride + i0;
    for (unsigned i = tid; i < wlen; i += kFirTile)
      s_a[i] = xa[i];
    if (MODE == 1)
    {
      const float* xb = p.inB + (size_t)s * p.in_stride + i0;
      for (unsigned i = tid; i < wlen; i += kFirTile)
        s_b[i] = xb[i];
    }
  }
  __syncthreads();
  for (unsigned t = tid; t < nt; t += kFirTile)
  {
    const unsigned i = i0 + t;
    const unsigned k0 = (p.g0 + i) % N;
    const unsigned base = (N - 1) + t; // window index of x[g]
    if (MODE == 2)
    {
      const float2* x = reinterpret_cast<const float2*>(s_a);
      float2 v = x[base - k0];
      float ar = mulf(s_coef[k0], v.x), ai = mulf(s_coef[k0], v.y);
#pragma unroll 4
      for (unsigned j = 1; j < N; ++j)
      {
        unsigned k = k0 + j;
        k = (k >= N) ? k - N : k;
        v = x[base - k];
        ar = addf(ar, mulf(s_coef[k], v.x));
        ai = addf(ai, mulf(s_coef[k], v.y));
      }
      reinterpret_cast<float2*>(p.outA)[(size_t)s * p.out_stride + p.out_off + i] = make_float2(ar, ai);
    }
    else
    {
      float a = mulf(s_coef[k0], s_a[base - k0]);
      float b = (MODE == 1) ? mulf(s_coef[k0], s_b[base - k0]) : 0.0f;
#pragma unroll 4
      for (unsigned j = 1; j < N; ++j)
      {
        unsigned k = k0 + j;
        k = (k >= N) ? k - N : k;
        const float c = s_coef[k];
        a = addf(a, mulf(c, s_a[base - k]));
        if (MODE == 1)
          b = addf(b, mulf(c, s_b[base - k]));
      }
      p.outA[(size_t)s * p.out_stride + p.out_off + i] = a;
      if (MODE == 1)
        p.outB[(size_t)s * p.out_stride + p.out_off + i] = b;
    }
  }
}

// --------------------------------------------------------------------------------------------------
// Lane = stream form of the same filter.  All streams of a decoder are in lock step, so the rotation
// k0 = (g0 + i) mod N of output i is the same for the 32 streams of a warp: taps become warp-uniform (one broadcast
// LDS), no per-lane modulo, and four consecutive outputs i .. i+3 whose rotations k0 .. k0+3 do not wrap share their
// samples.  Output i + r walks taps k0+r .. N-1 and then 0 .. k0+r-1 (the reference's buffer order), i.e. samples
//   phase 1:  V[N-1 + i - k0 - m],  m = 0 .. N-1-k0-r     tap k0 + r + m
//   phase 2:  V[N-1 + i + r - k],   k = 0 .. k0+r-1       tap k
// so the four outputs read the same sample at the same phase-1 step m, output r just stops r steps earlier, and in
// phase 2 output r starts r samples later: both phases are a common main loop (one sample LDS + one new tap per
// step, 4 x (mul, add) per channel) plus a 3-step triangle.  Every output receives exactly the reference's
// products in the reference's order (FirFilter.cpp:330-413) -- no zero padding, nothing reassociated.
// A CTA covers 32 streams x `cyc` whole rotation cycles (N outputs each, cut in G = g0 + i space so that groups of
// four never straddle a wrap); leftovers (N mod 4 outputs per cycle, block edges) take the one-output path.
// --------------------------------------------------------------------------------------------------
constexpr unsigned kRlWarps = 4;

template <int MODE, bool FUSED> // 0 real, 1 real pair, 2 complex
__global__ void __launch_bounds__(32 * kRlWarps) k_rotfir_lanes(RotFirParams p, unsigned cyc, unsigned pitch)
{
  extern __shared__ __align__(16) float rl_smem[];
  float* s_h = rl_smem;                                  // [N + 4]
  float* X = rl_smem + ((p.taps + 4 + 3) & ~3u);         // MODE 0: [32][pitch]; 1: [2][32][pitch]; 2: float2 [32][pitch]
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  const int N = (int)p.taps;
  const unsigned s0 = blockIdx.y * 32;
  const unsigned rows = min(32u, p.S - s0);
  // tile = cycles [blockIdx.x * cyc, +cyc) counted from the cycle that holds output 0
  const int ia_raw = (int)(blockIdx.x * cyc) * N - (int)(p.g0 % (unsigned)N);
  const int ia = max(ia_raw, 0), ib = min(ia_raw + (int)cyc * N, (int)p.n);
  if (ia >= ib)
    return;
  for (int i = tid; i < N + 4; i += 32 * kRlWarps)
    s_h[i] = i < N ? p.coef[i] : 0.0f;
  const int wlen = ib - ia + N - 1; // V[ia .. ia + wlen)
  // stage the window: a warp owns rows warp, warp + 4, ... (8 of them) and loads the same column of ALL its rows before
  // storing any (eight independent loads in flight per lane: the tile load is latency-bound, 28 % of the kernel's
  // stalls when the rows went one after the other)
  {
    constexpr int RW = 32 / kRlWarps;
    // element offsets of this warp's rows (32-bit: the address arithmetic of 16 loads per trip was 3/4 of this loop)
    unsigned roff[RW];
#pragma unroll
    for (int j = 0; j < RW; ++j)
      roff[j] = (s0 + min(warp + kRlWarps * j, rows - 1)) * (unsigned)p.in_stride + (unsigned)ia;
    for (int c = lane; c < wlen; c += 32)
    {
      if (MODE == 2)
      {
        float2 v[RW];
#pragma unroll
        for (int j = 0; j < RW; ++j)
        {
          const unsigned r = warp + kRlWarps * j;
          if (r < rows)
            v[j] = reinterpret_cast<const float2*>(p.inA)[roff[j] + (unsigned)c];
        }
#pragma unroll
        for (int j = 0; j < RW; ++j)
        {
          const unsigned r = warp + kRlWarps * j;
          if (r < rows)
            (reinterpret_cast<float2*>(X) + (size_t)r * pitch)[c] = v[j];
        }
      }
      else
      {
        float va[RW], vb[RW];
#pragma unroll
        for (int j = 0; j < RW; ++j)
        {
          const unsigned r = warp + kRlWarps * j;
          if (r < rows)
          {
            va[j] = p.inA[roff[j] + (unsigned)c];
            if (MODE == 1)
              vb[j] = p.inB[roff[j] + (unsigned)c];
          }
        }
#pragma unroll
        for (int j = 0; j < RW; ++j)
        {
          const unsigned r = warp + kRlWarps * j;
          if (r < rows)
          {
            // the two channels of a pair are kept interleaved: one 64-bit load per step instead of two 32-bit ones
            // (MODE 1 spent more instructions on addressing and loads than on arithmetic: 45 % FMUL / FADD)
            if (MODE == 1)
              (reinterpret_cast<float2*>(X) + (size_t)r * pitch)[c] = make_float2(va[j], vb[j]);
            else
              (X + (size_t)r * pitch)[c] = va[j];
          }
        }
      }
    }
  }
  __syncthreads();
  if (lane >= rows)
    return;
  const float* xa = X + (size_t)lane * pitch;
  const float2* xc = reinterpret_cast<const float2*>(X) + (size_t)lane * pitch;
  auto ld = [&](int col) -> float2 {
    if (MODE != 0)
      return xc[col];
    return make_float2(xa[col], 0.0f);
  };
  constexpr bool TWO = MODE != 0;
  const int gpc = (N + 3) / 4;
  const int total = (int)cyc * gpc;
  for (int gi = warp; gi < total; gi += kRlWarps)
  {
    const int cy = gi / gpc;
    const int k0 = (gi - cy * gpc) * 4;
    const int R = min(4, N - k0);
    const int i0 = ia_raw + cy * N + k0; // output index of r = 0
    if (R == 4 && i0 >= ia && i0 + 3 < ib)
    {
      const int col0 = i0 - ia + N - 1; // column of V[N-1 + i0]
      float2 a0, a1, a2, a3;
      float w0 = s_h[k0], w1 = s_h[k0 + 1], w2 = s_h[k0 + 2], w3 = s_h[k0 + 3];
      const int M1 = N - k0 - 3;
      int col = col0 - k0;
      {
        const float2 x = ld(col);
        a0.x = mulf(w0, x.x); a1.x = mulf(w1, x.x); a2.x = mulf(w2, x.x); a3.x = mulf(w3, x.x);
        if (TWO) { a0.y = mulf(w0, x.y); a1.y = mulf(w1, x.y); a2.y = mulf(w2, x.y); a3.y = mulf(w3, x.y); }
      }
#define RL_STEP4(x)                                                                                           \
  a0.x = macf<FUSED>(a0.x, w0, (x).x); a1.x = macf<FUSED>(a1.x, w1, (x).x);                                     \
  a2.x = macf<FUSED>(a2.x, w2, (x).x); a3.x = macf<FUSED>(a3.x, w3, (x).x);                                     \
  if (TWO) { a0.y = macf<FUSED>(a0.y, w0, (x).y); a1.y = macf<FUSED>(a1.y, w1, (x).y);                          \
             a2.y = macf<FUSED>(a2.y, w2, (x).y); a3.y = macf<FUSED>(a3.y, w3, (x).y); }
#pragma unroll 4
      for (int m = 1; m < M1; ++m)
      {
        w0 = w1; w1 = w2; w2 = w3; w3 = s_h[k0 + m + 3];
        const float2 x = ld(col - m);
        RL_STEP4(x)
      }
      col -= M1;
      { // phase-1 triangle: taps (N-3, N-2, N-1), (N-2, N-1), (N-1) = (w1, w2, w3), (w2, w3), (w3)
        float2 x = ld(col);
        a0.x = macf<FUSED>(a0.x, w1, (x).x); a1.x = macf<FUSED>(a1.x, w2, (x).x); a2.x = macf<FUSED>(a2.x, w3, (x).x);
        if (TWO) { a0.y = macf<FUSED>(a0.y, w1, (x).y); a1.y = macf<FUSED>(a1.y, w2, (x).y); a2.y = macf<FUSED>(a2.y, w3, (x).y); }
        x = ld(col - 1);
        a0.x = macf<FUSED>(a0.x, w2, (x).x); a1.x = macf<FUSED>(a1.x, w3, (x).x);
        if (TWO) { a0.y = macf<FUSED>(a0.y, w2, (x).y); a1.y = macf<FUSED>(a1.y, w3, (x).y); }
        x = ld(col - 2);
        a0.x = macf<FUSED>(a0.x, w3, (x).x);
        if (TWO) { a0.y = macf<FUSED>(a0.y, w3, (x).y); }
      }
      w0 = s_h[0]; w1 = s_h[1]; w2 = s_h[2]; w3 = s_h[3];
      { // phase-2 triangle: samples V[N-1 + i0 + 3], + 2, + 1
        float2 x = ld(col0 + 3);
        a3.x = macf<FUSED>(a3.x, w0, (x).x);
        if (TWO) { a3.y = macf<FUSED>(a3.y, w0, (x).y); }
        x = ld(col0 + 2);
        a2.x = macf<FUSED>(a2.x, w0, (x).x); a3.x = macf<FUSED>(a3.x, w1, (x).x);
        if (TWO) { a2.y = macf<FUSED>(a2.y, w0, (x).y); a3.y = macf<FUSED>(a3.y, w1, (x).y); }
        x = ld(col0 + 1);
        a1.x = macf<FUSED>(a1.x, w0, (x).x); a2.x = macf<FUSED>(a2.x, w1, (x).x); a3.x = macf<FUSED>(a3.x, w2, (x).x);
        if (TWO) { a1.y = macf<FUSED>(a1.y, w0, (x).y); a2.y = macf<FUSED>(a2.y, w1, (x).y); a3.y = macf<FUSED>(a3.y, w2, (x).y); }
      }
#pragma unroll 4
      for (int u = 0; u < k0; ++u)
      {
        const float2 x = ld(col0 - u);
        RL_STEP4(x)
        w0 = w1; w1 = w2; w2 = w3; w3 = s_h[u + 4];
      }
#undef RL_STEP4
      const size_t o = (size_t)(s0 + lane) * p.out_stride + p.out_off + (unsigned)i0;
      if (MODE == 2)
      {
        float2* out = reinterpret_cast<float2*>(p.outA) + o;
        out[0] = a0; out[1] = a1; out[2] = a2; out[3] = a3;
      }
      else
      {
        p.outA[o] = a0.x; p.outA[o + 1] = a1.x; p.outA[o + 2] = a2.x; p.outA[o + 3] = a3.x;
        if (MODE == 1)
        {
          p.outB[o] = a0.y; p.outB[o + 1] = a1.y; p.outB[o + 2] = a2.y; p.outB[o + 3] = a3.y;
        }
      }
      continue;
    }
    for (int r = 0; r < R; ++r)
    {
      const int i = i0 + r;
      if (i < ia || i >= ib)
        continue;
      const int kr = k0 + r;
      const int colx = i - ia + N - 1;
      float2 x = ld(colx - kr);
      float c = s_h[kr];
      float2 a;
      a.x = mulf(c, x.x);
      a.y = TWO ? mulf(c, x.y) : 0.0f;
      int k = kr;
      for (int j = 1; j < N; ++j)
      {
        k = (k + 1 == N) ? 0 : k + 1;
        x = ld(colx - k);
        c = s_h[k];
        a.x = addf(a.x, mulf(c, x.x));
        if (TWO)
          a.y = addf(a.y, mulf(c, x.y));
      }
      const size_t o = (size_t)(s0 + lane) * p.out_stride + p.out_off + (unsigned)i;
      if (MODE == 2)
        reinterpret_cast<float2*>(p.outA)[o] = a;
      else
      {
        p.outA[o] = a.x;
        if (MODE == 1)
          p.outB[o] = a.y;
      }
    }
  }
}

template <int MODE>
static void launch_rotfir_lanes(const RotFirParams& p, cudaStream_t st)
{
  const unsigned N = p.taps;
  static const unsigned target = (unsigned)KnobInt(RFM_KNOB("RFM_ROTFIR_OUT"), 128u); // measurement aid
  const unsigned cyc = std::max(1u, (target + N / 2) / N); // ~128 outputs per CTA
  const unsigned pitch = (cyc * N + N - 1) | 1u;        // odd: lanes (rows) hit distinct banks
  const size_t smem = (((N + 4 + 3) & ~3u) + (size_t)(MODE == 0 ? 1 : 2) * 32 * pitch) * sizeof(float);
  const unsigned cycles = (p.g0 % N + p.n + N - 1) / N;
  dim3 grid(cdiv(cycles, cyc), cdiv(p.S, 32));
  if (p.fused)
  {
    EnsureDynSmem(k_rotfir_lanes<MODE, true>, smem);
    k_rotfir_lanes<MODE, true><<<grid, 32 * kRlWarps, smem, st>>>(p, cyc, pitch);
  }
  else
  {
    EnsureDynSmem(k_rotfir_lanes<MODE, false>, smem);
    k_rotfir_lanes<MODE, false><<<grid, 32 * kRlWarps, smem, st>>>(p, cyc, pitch);
  }
}

void launch_rotfir(const RotFirParams& p, cudaStream_t st)
{
  if (p.n == 0 || p.S == 0)
    return;
  static const bool old_form = RFM_KNOB("RFM_ROTFIR_OLD") != nullptr; // measurement aid
  if (p.taps >= 8 && !old_form)
  {
    if (p.cplx)
      launch_rotfir_lanes<2>(p, st);
    else if (p.inB)
      launch_rotfir_lanes<1>(p, st);
    else
      launch_rotfir_lanes<0>(p, st);
    return;
  }
  dim3 grid(cdiv(p.n, kFirOut), p.S);
  if (p.cplx)
    k_rotfir<2><<<grid, kFirTile, 0, st>>>(p);
  else if (p.inB)
    k_rotfir<1><<<grid, kFirTile, 0, st>>>(p);
  else
    k_rotfir<0><<<grid, kFirTile, 0, st>>>(p);
}

// ==================================================================================================
// audio tail lanes: deemphasis (FmDecode.cpp:348-359), notch (IirFilter.cpp:89-105),
// matrix (FmDecode.cpp:473-499)
// ==================================================================================================
struct AudioTailSmem
{
  float inS[2][32][kLT + 1];
  float inM[2][32][kLT + 1];
  float2 out[32][kLT + 1];
};

__global__ void __launch_bounds__(32) k_audio_tail(AudioTailParams p)
{
  __shared__ AudioTailSmem sm;
  const unsigned lane = threadIdx.x;
  const unsigned s0 = blockIdx.x * 32;
  const unsigned s = s0 + lane;
  const bool valid = s < p.S;
  const unsigned S = p.S;
  float* st = p.state;
  float de_re = 0.f, de_im = 0.f, w1a = 0.f, w2a = 0.f, w1b = 0.f, w2b = 0.f;
  bool stereo = false;
  if (valid)
  {
    de_re = st[SF_DE_RE * S + s]; de_im = st[SF_DE_IM * S + s];
    w1a = st[SF_NOTCH_W1A * S + s]; w2a = st[SF_NOTCH_W2A * S + s];
    w1b = st[SF_NOTCH_W1B * S + s]; w2b = st[SF_NOTCH_W2B * S + s];
    stereo = __float_as_int(st[(SF_STEREO + p.parity) * S + s]) != 0;
  }
  const float alpha = p.de_alpha;
  const float one_m = subf(1.0f, alpha);
  const unsigned ntiles = (p.na + kLT - 1) / kLT;
  tile_load_async(sm.inS[0], p.inS, p.in_stride, s0, S, 0, p.na, lane);
  tile_load_async(sm.inM[0], p.inM, p.in_stride, s0, S, 0, p.na, lane);
  cp_async_commit();
  for (unsigned t = 0; t < ntiles; ++t)
  {
    const unsigned b = t & 1u, t0 = t * kLT;
    const unsigned tn = min(kLT, p.na - t0);
    if (t + 1 < ntiles)
    {
      tile_load_async(sm.inS[b ^ 1u], p.inS, p.in_stride, s0, S, t0 + kLT, p.na, lane);
      tile_load_async(sm.inM[b ^ 1u], p.inM, p.in_stride, s0, S, t0 + kLT, p.na, lane);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    if (valid)
    {
      for (unsigned k = 0; k < tn; ++k)
      {
        de_re = addf(mulf(one_m, de_re), mulf(alpha, sm.inS[b][lane][k]));
        const float a = mulf(de_re, 2.0f);
        de_im = addf(mulf(one_m, de_im), mulf(alpha, sm.inM[b][lane][k]));
        const float bm = mulf(de_im, 2.0f);
        const float sd = biquad_step(p.notch, a, w1a, w2a);
        const float m = biquad_step(p.notch, bm, w1b, w2b);
        float2 o;
        if (stereo)
        {
          o.x = mulf(addf(m, sd), 0.5f);
          o.y = mulf(subf(m, sd), 0.5f);
        }
        else
        {
          o.x = mulf(m, 0.5f);
          o.y = o.x;
        }
        sm.out[lane][k] = o;
      }
    }
    __syncwarp();
    tile_store(reinterpret_cast<float2*>(p.audio), p.audio_stride / 2, s0, S, t0, p.na, lane, sm.out);
    __syncwarp();
  }
  if (valid)
  {
    st[SF_DE_RE * S + s] = de_re;
    st[SF_DE_IM * S + s] = de_im;
    st[SF_NOTCH_W1A * S + s] = w1a;
    st[SF_NOTCH_W2A * S + s] = w2a;
    st[SF_NOTCH_W1B * S + s] = w1b;
    st[SF_NOTCH_W2B * S + s] = w2b;
  }
}

void launch_audio_tail(const AudioTailParams& p, cudaStream_t st)
{
  if (p.S == 0 || p.na == 0)
    return;
  k_audio_tail<<<cdiv(p.S, 32), 32, 0, st>>>(p);
}

// ==================================================================================================
// RDS: NCO_OSC table, DownConvert.cpp:438-442 -- identical for every stream of the decoder
// ==================================================================================================
__global__ void k_osc(OscParams p)
{
  if (threadIdx.x != 0 || blockIdx.x != 0)
    return;
  float o1r = p.osc1[0], o1i = p.osc1[1];
  float2* out = reinterpret_cast<float2*>(p.oscV) + p.osc_hist;
  for (unsigned i = 0; i < p.nb; ++i)
  {
    const float orr = subf(mulf(o1r, p.cosv), mulf(o1i, p.sinv));
    const float oi = addf(mulf(o1i, p.cosv), mulf(o1r, p.sinv));
    const float gn = rfm_osc_gain(addf(mulf(o1r, o1r), mulf(o1i, o1i))); // == float(1.95 - double(q)), rfm_dsp.cuh
    o1r = mulf(gn, orr);
    o1i = mulf(gn, oi);
    out[i] = make_float2(orr, oi);
  }
  p.osc1[0] = o1r;
  p.osc1[1] = o1i;
}

void launch_osc(const OscParams& p, cudaStream_t st)
{
  if (p.nb == 0)
    return;
  k_osc<<<1, 32, 0, st>>>(p);
}

// ==================================================================================================
// RDS branch: decimate-by-2 stages, DownConvert.cpp:516-550 (generic), :589-688 (11-tap), :709-727 (CIC3)
// ==================================================================================================
// --------------------------------------------------------------------------------------------------
// Fused RDS front: NCO mix (DownConvert.cpp:438-442,464-465) -> every decimate-by-2 stage (:516-550, :589-688,
// :709-727) -> the 2.4 kHz Kaiser LP (cFirFilter::Process complex, FirFilter.cpp:330-350; RDSProcess.cpp:128).
// One CTA per stream walks the block in tiles of kRfTile baseband samples; every stage lives in a shared-memory
// "V buffer" [history | tile], so no intermediate ever goes to HBM (the unfused chain wrote and re-read 4 of them).
// Histories are carried tile to tile in shared memory and block to block in a small per-stream tail row.
// Arithmetic and summation orders are those of k_halfband / k_rotfir (bit-identical results).
// --------------------------------------------------------------------------------------------------
constexpr unsigned kRfTile = 1024;
constexpr unsigned kRfThreads = 128;

__global__ void __launch_bounds__(kRfThreads) k_rds_front(RdsFrontParams p)
{
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // layout: taps of every stage, LP taps, then the V buffers of stage 0 .. nst-1 and of the LP
  float* s_h = reinterpret_cast<float*>(smem_raw);
  // per-stage descriptors in SHARED memory: the stage loops index them with a run-time k, and as local arrays they
  // lived on the stack (88 bytes of local memory, a long-scoreboard stall per access: 26 % of this kernel's stalls)
  __shared__ unsigned s_hoff[kRfMaxStages + 1], s_boff[kRfMaxStages + 1], s_len[kRfMaxStages], s_hist[kRfMaxStages + 1],
      s_kind[kRfMaxStages], s_lpoff[2];
  if (threadIdx.x == 0)
  {
    unsigned acc = 0, off = 0, n = kRfTile;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      s_hoff[k] = acc;
      acc += (p.st[k].len + 1u) & ~1u;
      s_len[k] = p.st[k].len;
      s_hist[k] = p.st[k].hist;
      s_kind[k] = (unsigned)p.st[k].kind;
    }
    s_hoff[p.nst] = acc;
    s_hist[p.nst] = p.lp_n - 1;
    s_lpoff[0] = acc;
    acc += (p.lp_n + 1u) & ~1u;
    s_lpoff[1] = acc;
    for (unsigned k = 0; k <= p.nst; ++k)
    {
      s_boff[k] = off;
      off += s_hist[k] + n;
      n >>= 1;
    }
  }
  __syncthreads();
  float* s_lp = s_h + s_lpoff[0];
  float2* vbuf = reinterpret_cast<float2*>(s_h + s_lpoff[1]);
#define RFM_B(k) (vbuf + s_boff[k])
  const unsigned tid = threadIdx.x;
  const unsigned s = blockIdx.x;
  for (unsigned k = 0; k < p.nst; ++k)
    for (unsigned i = tid; i < s_len[k]; i += kRfThreads)
      s_h[s_hoff[k] + i] = p.st[k].h ? p.st[k].h[i] : 0.0f;
  for (unsigned i = tid; i < p.lp_n; i += kRfThreads)
    s_lp[i] = p.lp_coef[i];
  // histories from the previous block
  const bool ext_lp = p.lp_v != nullptr;           // the LP runs as its own kernel on lp_v
  const unsigned nbuf = ext_lp ? p.nst : p.nst + 1; // V buffers with a carried history
  float2* lpv = ext_lp ? reinterpret_cast<float2*>(p.lp_v) + (size_t)blockIdx.x * p.lp_v_stride + (p.lp_n - 1) : nullptr;
  float2* tails = reinterpret_cast<float2*>(p.tails) + (size_t)s * p.tail_stride;
  for (unsigned k = 0; k < nbuf; ++k)
  {
    const unsigned hist = s_hist[k];
    for (unsigned i = tid; i < hist; i += kRfThreads)
      RFM_B(k)[i] = tails[p.tail_off[k] + i];
  }
  __syncthreads();

  const float* bb = p.bbV + (size_t)s * p.a_stride + p.a_hist;
  const float2* osc = reinterpret_cast<const float2*>(p.osc);
  float2* out = reinterpret_cast<float2*>(p.out) + (size_t)s * p.out_stride;
  const unsigned N = p.lp_n;
  unsigned out_base = 0; // LP outputs produced so far in this block
  // the baseband / oscillator samples of the NEXT tile travel to shared memory (cp.async) while the stages of the
  // current one run: the tile loads were this kernel's largest stall
  float* s_bbst;
  float2* s_oscst;
  {
    unsigned n = kRfTile >> p.nst;
    s_oscst = vbuf + s_boff[p.nst] + s_hist[p.nst] + n;
    s_bbst = reinterpret_cast<float*>(s_oscst + kRfTile);
  }
  auto stage_tile = [&](unsigned t0n) {
    const unsigned tnn = min(kRfTile, p.nb - t0n);
    for (unsigned i = tid; i < tnn; i += kRfThreads)
    {
      cp_async_4(&s_bbst[i], &bb[t0n + i]);
      cp_async_8(&s_oscst[i], &osc[t0n + i]);
    }
    cp_async_commit();
  };
  stage_tile(0);
  for (unsigned t0 = 0; t0 < p.nb; t0 += kRfTile)
  {
    const unsigned tn = min(kRfTile, p.nb - t0);
    cp_async_wait<0>();
    __syncthreads();
    // mix: real baseband x NCO phasor, imaginary input exactly +0 (RDSProcess.cpp:122-123)
    for (unsigned i = tid; i < tn; i += kRfThreads)
    {
      const float b = s_bbst[i];
      const float2 o = s_oscst[i];
      float2 r;
      r.x = subf(mulf(b, o.x), mulf(0.0f, o.y));
      r.y = addf(mulf(b, o.y), mulf(0.0f, o.x));
      RFM_B(0)[s_hist[0] + i] = r;
    }
    __syncthreads();
    if (t0 + kRfTile < p.nb)
      stage_tile(t0 + kRfTile);
    unsigned n = tn;
    for (unsigned k = 0; k < p.nst; ++k)
    {
      // an odd count (generic half-band only: the host plans it) makes (n + 1) / 2 outputs, the last one ending on the
      // newest sample; a stage that is SHORT this block passes the first n / 2 inputs through (DownConvert.cpp:498-550)
      const bool shortk = (p.short_mask >> k) & 1u;
      const unsigned nout = shortk ? (n >> 1) : ((n + 1) >> 1);
      const unsigned ohist = s_hist[k + 1];
      const unsigned kind = s_kind[k], len = s_len[k];
      const float* hk = s_h + s_hoff[k];
      const float2* bin = RFM_B(k);
      float2* bout = RFM_B(k + 1);
      const bool last = (k + 1 == p.nst) && p.dec_out != nullptr;
      const bool to_lpv = (k + 1 == p.nst) && ext_lp;
      for (unsigned o = tid; o < nout; o += kRfThreads)
      {
        const float2 v = shortk ? bin[s_hist[k] + o] : hb_out((int)kind, len, hk, bin, o);
        if (to_lpv)
          lpv[out_base + o] = v;
        else
          bout[ohist + o] = v;
        if (last) // decimator output (cRDSRxSignalProcessor's m_RdsRaw before the LP), kept for the stage taps
          reinterpret_cast<float2*>(p.dec_out)[(size_t)s * p.out_stride + out_base + o] = v;
      }
      __syncthreads();
      n = nout;
    }
    // LP with cFirFilter's rotating summation start: y[g] = sum_j h[k_j] x[g - k_j], k_j = (g + j) mod N
    for (unsigned i = tid; i < n && !ext_lp; i += kRfThreads)
    {
      unsigned k = (p.g0 + out_base + i) % N;
      const float2* x = RFM_B(p.nst) + (N - 1) + i;
      float2 v = x[-(int)k];
      float ar = mulf(s_lp[k], v.x), ai = mulf(s_lp[k], v.y);
      // uniform trip count (the start tap differs per lane): wrap with a compare / select, no modulo
#pragma unroll 5
      for (unsigned j = 1; j < N; ++j)
      {
        unsigned q = k + j;
        q = (q >= N) ? q - N : q;
        v = x[-(int)q];
        ar = addf(ar, mulf(s_lp[q], v.x));
        ai = addf(ai, mulf(s_lp[q], v.y));
      }
      out[out_base + i] = make_float2(ar, ai);
    }
    out_base += n;
    __syncthreads();
    // carry the histories: last `hist` entries of [hist | n_k] to the front
    {
      unsigned nk = tn;
      for (unsigned k = 0; k < nbuf; ++k)
      {
        const bool shortk = k < p.nst && ((p.short_mask >> k) & 1u); // a short stage keeps its delay line
        const unsigned hist = shortk ? 0u : s_hist[k];
        float2* bk = RFM_B(k);
        float2 v0 = make_float2(0.f, 0.f);
        if (tid < hist)
          v0 = bk[nk + tid];
        __syncthreads();
        if (tid < hist)
          bk[tid] = v0;
        nk = shortk ? (nk >> 1) : ((nk + 1) >> 1);
      }
    }
    __syncthreads();
  }
  for (unsigned k = 0; k < nbuf; ++k)
  {
    const unsigned hist = s_hist[k];
    for (unsigned i = tid; i < hist; i += kRfThreads)
      tails[p.tail_off[k] + i] = RFM_B(k)[i];
  }
}
#undef RFM_B

// --------------------------------------------------------------------------------------------------
// Register-tiled RDS front for the plans the reference's caller produces at 1.0 / 1.2 / 2.4 MS/s: three generic
// half-band stages (HB15, HB19 | HB23, HB35 | HB43), the LP on its own kernel (lp_v).  Same fusion as k_rds_front --
// one CTA per stream walks the block in tiles, nothing intermediate in HBM -- but the stage buffers are kept
// DE-INTERLEAVED (rfm_dsp.cuh: hb_deint): a thread makes R consecutive outputs from registers and the taps are
// constant-bank operands, so an output costs (L+1)/2R + 1 shared-memory loads instead of one sample load AND one tap
// load per tap (k_rds_front ran at 85 % of the shared-memory pipe, 6.9 short-scoreboard stall cycles per issue).
// Arithmetic and summation order are those of hb_generic / DownConvert.cpp:528-540: bit-identical results.
// --------------------------------------------------------------------------------------------------
constexpr unsigned kRf3Tile = 1024;   // baseband samples per tile
constexpr unsigned kRf3Threads = 128;

template <int L, int R>
__device__ __forceinline__ void rf3_stage(const DcTapsPk<L>& taps, const float2* E, const float2* O, float2* dstE, float2* dstO,
                                          unsigned nout, unsigned tid)
{
  // dstO == nullptr: last stage, dstE is the output row (natural order); else output o goes to the next stage's
  // E / O by parity (both pre-offset by that stage's history).  Arithmetic on packed (re, im) pairs: hb_deint_pk
  for (unsigned g = tid; g * R < nout; g += kRf3Threads)
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

template <int L0, int L1, int L2>
__global__ void __launch_bounds__(kRf3Threads) k_rds_front3(RdsFrontParams p, DcTapsPk<L0> t0, DcTapsPk<L1> t1, DcTapsPk<L2> t2)
{
  constexpr unsigned T = kRf3Tile, SL = 6; // SL: slack behind each buffer (a group of R outputs may read past the tile)
  constexpr unsigned H0 = (L0 - 1) / 2, H1 = (L1 - 1) / 2, H2 = (L2 - 1) / 2; // history entries in each of E and O
  constexpr unsigned Z0 = (H0 + T / 2 + SL + 1) & ~1u, Z1 = (H1 + T / 4 + SL + 1) & ~1u, Z2 = (H2 + T / 8 + SL + 1) & ~1u;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* E0 = reinterpret_cast<float2*>(smem_raw);
  float2* O0 = E0 + Z0;
  float2* E1 = O0 + Z0;
  float2* O1 = E1 + Z1;
  float2* E2 = O1 + Z1;
  float2* O2 = E2 + Z2;
  float2* s_osc = O2 + Z2;                              // [T], 16-byte aligned (every Z is even)
  float* s_bb = reinterpret_cast<float*>(s_osc + T);    // [T]
  const unsigned tid = threadIdx.x;
  const unsigned s = blockIdx.x;
  float2* tails = reinterpret_cast<float2*>(p.tails) + (size_t)s * p.tail_stride;
  // histories from the previous block: V index i of stage k's [history | tile] row -> (i odd ? O : E)[i / 2]
  auto load_hist = [&](float2* E, float2* O, unsigned H, unsigned off) {
    for (unsigned i = tid; i < 2 * H; i += kRf3Threads)
      ((i & 1u) ? O : E)[i >> 1] = tails[off + i];
  };
  load_hist(E0, O0, H0, p.tail_off[0]);
  load_hist(E1, O1, H1, p.tail_off[1]);
  load_hist(E2, O2, H2, p.tail_off[2]);

  const float* bb = p.bbV + (size_t)s * p.a_stride + p.a_hist;
  const float2* osc = reinterpret_cast<const float2*>(p.osc);
  float2* lpv = reinterpret_cast<float2*>(p.lp_v) + (size_t)s * p.lp_v_stride + (p.lp_n - 1);
  auto stage_tile = [&](unsigned t0n) {
    const unsigned tnn = min(T, p.nb - t0n); // multiple of 8
    for (unsigned i = tid; 2 * i < tnn; i += kRf3Threads)
    {
      cp_async_8(&s_bb[2 * i], &bb[t0n + 2 * i]);
      cp_async_16(&s_osc[2 * i], &osc[t0n + 2 * i]);
    }
    cp_async_commit();
  };
  stage_tile(0);
  unsigned out_base = 0;
  for (unsigned tb = 0; tb < p.nb; tb += T)
  {
    const unsigned tn = min(T, p.nb - tb);
    cp_async_wait<0>();
    __syncthreads();
    // mix: real baseband x NCO phasor, imaginary input exactly +0 (RDSProcess.cpp:122-123); sample pairs -> E0 / O0
    for (unsigned i = tid; 2 * i < tn; i += kRf3Threads)
    {
      const float2 b = *reinterpret_cast<const float2*>(&s_bb[2 * i]);
      const float4 o = *reinterpret_cast<const float4*>(&s_osc[2 * i]);
      float2 e, d;
      e.x = subf(mulf(b.x, o.x), mulf(0.0f, o.y));
      e.y = addf(mulf(b.x, o.y), mulf(0.0f, o.x));
      d.x = subf(mulf(b.y, o.z), mulf(0.0f, o.w));
      d.y = addf(mulf(b.y, o.w), mulf(0.0f, o.z));
      E0[H0 + i] = e;
      O0[H0 + i] = d;
    }
    __syncthreads();
    if (tb + T < p.nb)
      stage_tile(tb + T);
    rf3_stage<L0, 5>(t0, E0, O0, E1 + H1, O1 + H1, tn >> 1, tid);
    __syncthreads();
    rf3_stage<L1, 3>(t1, E1, O1, E2 + H2, O2 + H2, tn >> 2, tid);
    __syncthreads();
    rf3_stage<L2, 1>(t2, E2, O2, lpv + out_base, nullptr, tn >> 3, tid);
    out_base += tn >> 3;
    // carry the histories: the last H entries of [H | n / 2] to the front, in each of E and O (memmove semantics: a
    // ragged last tile may be shorter than the history)
    {
      const float2 a0 = tid < H0 ? E0[(tn >> 1) + tid] : make_float2(0.f, 0.f);
      const float2 b0 = tid < H0 ? O0[(tn >> 1) + tid] : make_float2(0.f, 0.f);
      const float2 a1 = tid < H1 ? E1[(tn >> 2) + tid] : make_float2(0.f, 0.f);
      const float2 b1 = tid < H1 ? O1[(tn >> 2) + tid] : make_float2(0.f, 0.f);
      const float2 a2 = tid < H2 ? E2[(tn >> 3) + tid] : make_float2(0.f, 0.f);
      const float2 b2 = tid < H2 ? O2[(tn >> 3) + tid] : make_float2(0.f, 0.f);
      __syncthreads();
      if (tid < H0) { E0[tid] = a0; O0[tid] = b0; }
      if (tid < H1) { E1[tid] = a1; O1[tid] = b1; }
      if (tid < H2) { E2[tid] = a2; O2[tid] = b2; }
    }
    // (the next iteration's first barrier orders these writes before any reader)
  }
  __syncthreads();
  auto store_hist = [&](const float2* E, const float2* O, unsigned H, unsigned off) {
    for (unsigned i = tid; i < 2 * H; i += kRf3Threads)
      tails[off + i] = ((i & 1u) ? O : E)[i >> 1];
  };
  store_hist(E0, O0, H0, p.tail_off[0]);
  store_hist(E1, O1, H1, p.tail_off[1]);
  store_hist(E2, O2, H2, p.tail_off[2]);
}

template <int L0, int L1, int L2>
static void launch_rds_front3(const RdsFrontParams& p, cudaStream_t st)
{
  DcTaps<L0> t0;
  DcTaps<L1> t1;
  DcTaps<L2> t2;
  memcpy(t0.h, p.st[0].h_host, sizeof(t0.h));
  memcpy(t1.h, p.st[1].h_host, sizeof(t1.h));
  memcpy(t2.h, p.st[2].h_host, sizeof(t2.h));
  constexpr unsigned T = kRf3Tile, SL = 6;
  constexpr unsigned Z0 = ((L0 - 1) / 2 + T / 2 + SL + 1) & ~1u, Z1 = ((L1 - 1) / 2 + T / 4 + SL + 1) & ~1u,
                     Z2 = ((L2 - 1) / 2 + T / 8 + SL + 1) & ~1u;
  const size_t smem = (size_t)(2 * (Z0 + Z1 + Z2) + T) * sizeof(float2) + T * sizeof(float);
  EnsureDynSmem(k_rds_front3<L0, L1, L2>, smem);
  k_rds_front3<L0, L1, L2><<<p.S, kRf3Threads, smem, st>>>(p, MakeDcTapsPk(t0), MakeDcTapsPk(t1), MakeDcTapsPk(t2));
}

void launch_rds_front(const RdsFrontParams& p, cudaStream_t st)
{
  if (p.S == 0 || p.nb == 0)
    return;
  // the three-stage plans of the reference's caller (SURVEY.md section 8 table), LP on its own kernel
  if (p.nst == 3 && p.lp_v && !p.dec_out && p.nb % 8 == 0 && p.short_mask == 0 && p.st[0].kind == 0 && p.st[1].kind == 0 && p.st[2].kind == 0 &&
      p.st[0].h_host && p.st[1].h_host && p.st[2].h_host && (p.a_hist & 1u) == 0 && (p.a_stride & 1u) == 0 &&
      (reinterpret_cast<uintptr_t>(p.osc) & 15u) == 0 && (reinterpret_cast<uintptr_t>(p.bbV) & 7u) == 0)
  {
    const unsigned l0 = p.st[0].len, l1 = p.st[1].len, l2 = p.st[2].len;
    if (l0 == 15 && l1 == 23 && l2 == 43)
      return launch_rds_front3<15, 23, 43>(p, st);
    if (l0 == 15 && l1 == 19 && l2 == 35)
      return launch_rds_front3<15, 19, 35>(p, st);
  }
  size_t floats = 0;
  for (unsigned k = 0; k < p.nst; ++k)
    floats += (p.st[k].len + 1u) & ~1u;
  floats += (p.lp_n + 1u) & ~1u;
  size_t f2 = 0;
  unsigned n = kRfTile;
  for (unsigned k = 0; k <= p.nst; ++k)
  {
    f2 += ((k < p.nst) ? p.st[k].hist : p.lp_n - 1) + n;
    n >>= 1;
  }
  const size_t smem = floats * sizeof(float) + f2 * sizeof(float2) + kRfTile * (sizeof(float2) + sizeof(float)); // + tile staging
  EnsureDynSmem(k_rds_front, smem);
  k_rds_front<<<p.S, kRfThreads, smem, st>>>(p);
}

// ==================================================================================================
// RDS Costas loop, RDSProcess.cpp:187-270
// ==================================================================================================
struct RdsPllSmem
{
  float2 in[2][32][kLT + 1];
  float out[32][kLT + 1];
};

__global__ void __launch_bounds__(32) k_rds_pll(RdsPllParams p)
{
  __shared__ RdsPllSmem sm;
  const unsigned lane = threadIdx.x;
  const unsigned s0 = blockIdx.x * 32;
  const unsigned s = s0 + lane;
  const bool valid = s < p.S;
  const unsigned S = p.S;
  float phase = 0.f, freq = 0.f;
  if (valid)
  {
    phase = p.state[SF_RPLL_PHASE * S + s];
    freq = p.state[SF_RPLL_FREQ * S + s];
  }
  const float2* in = reinterpret_cast<const float2*>(p.in);
  const unsigned ntiles = (p.nr + kLT - 1) / kLT;
  tile_load_async(sm.in[0], in, p.in_stride, s0, S, 0, p.nr, lane);
  cp_async_commit();
  for (unsigned t = 0; t < ntiles; ++t)
  {
    const unsigned b = t & 1u, t0 = t * kLT;
    const unsigned tn = min(kLT, p.nr - t0);
    if (t + 1 < ntiles)
      tile_load_async(sm.in[b ^ 1u], in, p.in_stride, s0, S, t0 + kLT, p.nr, lane);
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    if (valid)
    {
      for (unsigned k = 0; k < tn; ++k)
      {
        const float2 x = sm.in[b][lane][k];
        sm.out[lane][k] = rds_pll_step(phase, freq, x.x, x.y, p.lo, p.hi, p.alpha, p.beta);
      }
    }
    __syncwarp();
    tile_store(p.out + p.out_off, p.out_stride, s0, S, t0, p.nr, lane, sm.out);
    __syncwarp();
  }
  if (valid)
  {
    phase = rfm_fmodf_small(phase, d2f(RFM_K_2PI)); // RDSProcess.cpp:269
    p.state[SF_RPLL_PHASE * S + s] = phase;
    p.state[SF_RPLL_FREQ * S + s] = freq;
  }
}

void launch_rds_pll(const RdsPllParams& p, cudaStream_t st)
{
  if (p.S == 0 || p.nr == 0)
    return;
  k_rds_pll<<<cdiv(p.S, 32), 32, 0, st>>>(p);
}

// ==================================================================================================
// bit clock + slicer, RDSProcess.cpp:137-179
// ==================================================================================================
__global__ void __launch_bounds__(32) k_rds_slice(RdsSliceParams p)
{
  __shared__ float tin[2][32][kLT + 1];
  const unsigned lane = threadIdx.x;
  const unsigned s0 = blockIdx.x * 32;
  const unsigned s = s0 + lane;
  const bool valid = s < p.S;
  const unsigned S = p.S;
  float* st = p.state;
  float w1 = 0.f, w2 = 0.f, last_sync = 0.f, last_slope = 0.f, last_data = 0.f;
  int last_bit = 0;
  unsigned cnt = 0;
  if (valid)
  {
    w1 = st[SF_RSYNC_W1 * S + s]; w2 = st[SF_RSYNC_W2 * S + s];
    last_sync = st[SF_RS_LASTSYNC * S + s]; last_slope = st[SF_RS_LASTSLOPE * S + s];
    last_data = st[SF_RS_LASTDATA * S + s];
    last_bit = __float_as_int(st[SF_RS_LASTBIT * S + s]);
    cnt = p.bit_count[s];
  }
  uint8_t* bits = p.bits + (size_t)s * p.bits_cap;
  const unsigned ntiles = (p.nr + kLT - 1) / kLT;
  tile_load_async(tin[0], p.in, p.in_stride, s0, S, 0, p.nr, lane);
  cp_async_commit();
  for (unsigned t = 0; t < ntiles; ++t)
  {
    const unsigned b = t & 1u, t0 = t * kLT;
    const unsigned tn = min(kLT, p.nr - t0);
    if (t + 1 < ntiles)
      tile_load_async(tin[b ^ 1u], p.in, p.in_stride, s0, S, t0 + kLT, p.nr, lane);
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    if (valid)
    {
      for (unsigned k = 0; k < tn; ++k)
      {
        const float d = tin[b][lane][k];
        const float mag = mulf(d, d);
        const float sync = biquad_step(p.sync, mag, w1, w2);
        const float slope = subf(sync, last_sync);
        last_sync = sync;
        if (slope < 0.0f && mulf(last_slope, slope) < 0.0f)
        {
          const int bit = (last_data >= 0.0f) ? 1 : 0;
          if (cnt < p.bits_cap)
            bits[cnt] = (uint8_t)(bit ^ last_bit);
          ++cnt;
          last_bit = bit;
        }
        last_data = d;
        last_slope = slope;
      }
    }
    __syncwarp();
  }
  if (valid)
  {
    p.bit_count[s] = cnt;
    st[SF_RSYNC_W1 * S + s] = w1;
    st[SF_RSYNC_W2 * S + s] = w2;
    st[SF_RS_LASTSYNC * S + s] = last_sync;
    st[SF_RS_LASTSLOPE * S + s] = last_slope;
    st[SF_RS_LASTDATA * S + s] = last_data;
    st[SF_RS_LASTBIT * S + s] = __int_as_float(last_bit);
  }
}

void launch_rds_slice(const RdsSliceParams& p, cudaStream_t st)
{
  if (p.S == 0 || p.nr == 0)
    return;
  k_rds_slice<<<cdiv(p.S, 32), 32, 0, st>>>(p);
}

// ==================================================================================================
// history carry: row = [hist | n]  ->  first `hist` elements := last `hist` elements
// ==================================================================================================
template <typename T>
__device__ __forceinline__ void tail_row(const T* row, T* dst, unsigned hist, unsigned n)
{
  // hist <= 2 * blockDim.x (checked on the host); values are read before any is written, so the
  // overlapping case n < hist is handled too (memmove semantics).
  T v0, v1;
  const unsigned a = threadIdx.x, b = threadIdx.x + blockDim.x;
  if (a < hist)
    v0 = row[n + a];
  if (b < hist)
    v1 = row[n + b];
  __syncthreads();
  if (a < hist)
    dst[a] = v0;
  if (b < hist)
    dst[b] = v1;
}

__global__ void __launch_bounds__(256) k_tails(TailParams p)
{
  const TailDesc d = p.d[blockIdx.y];
  if (blockIdx.x >= d.rows)
    return;
  const unsigned char* row = reinterpret_cast<const unsigned char*>(d.base) + (size_t)blockIdx.x * d.stride_bytes;
  unsigned char* dst = reinterpret_cast<unsigned char*>(d.dst) + (size_t)blockIdx.x * d.stride_bytes;
  if (d.elem == 8)
    tail_row(reinterpret_cast<const uint2*>(row), reinterpret_cast<uint2*>(dst), d.hist, d.n);
  else
    tail_row(reinterpret_cast<const uint32_t*>(row), reinterpret_cast<uint32_t*>(dst), d.hist, d.n);
}

void launch_tails(const TailParams& p, unsigned S, cudaStream_t st)
{
  if (p.count == 0 || S == 0)
    return;
  dim3 grid(S, p.count);
  k_tails<<<grid, 256, 0, st>>>(p);
}

} // namespace rfm
