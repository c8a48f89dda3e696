// rfm_iqcorr.cu -- blind estimate of the frequency-flat IQ correction of a capture (rfm_iq_correction,
// include/radiofm_b200.h): the DC offset and the gain / phase imbalance of a zero-IF receiver.  One read of the capture:
//
//   k_iq_stats<F>      CTA b sums samples [b * kStChunk, (b + 1) * kStChunk): S_I, S_Q, S_II, S_QQ, S_IQ, one partial
//                      row per CTA.  u8 / s8 / s16: integer codes, 64-bit integer sums (exact: any order gives the same
//                      value).  cf32: double sums, each thread over a fixed stride, then a fixed shuffle tree and the
//                      warps in order -- the order depends on n only.
//   k_iq_stats_reduce  the partial rows summed in a fixed order (thread t takes rows t, t + 256, ..; then thread 0 sums
//                      the 256 results in order), no atomics.
//
// The coefficients are computed on the host from the five sums (IqCoefficients): centred moments n S_xy - S_x S_y in
// 128-bit integers for the integer formats, then every value in double, rounded to float once.  oracle/iqcorr.py
// evaluates the same expressions in the same order, so integer-format coefficients are bit-identical to it.
// The correction itself is applied inside the kernels that convert the capture (rfm_iq_correct, rfm_dsp.cuh).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <atomic>
#include <string>

#include "../../include/radiofm_b200.h"
#include "rfm_dsp.cuh"

namespace rfm
{
extern std::atomic<uint64_t> g_launches;
void SetLastError(const std::string& m);
}

namespace
{
using namespace rfm;

constexpr unsigned kStThreads = 256;
constexpr unsigned kStPerThread = 64;
constexpr unsigned kStChunk = kStThreads * kStPerThread;   // samples per CTA, fixed: the split depends on n only
constexpr unsigned kStSums = 5;                              // S_I, S_Q, S_II, S_QQ, S_IQ

template <int F> struct StAcc { using T = long long; };
template <> struct StAcc<kIqCF32> { using T = double; };

// integer codes of sample i (u8: 0..255, s8: -128..127, s16: -32768..32767)
template <int F>
__device__ __forceinline__ void st_codes(const void* in, uint64_t i, int& I, int& Q)
{
  if (F == kIqS16)
  {
    const unsigned w = reinterpret_cast<const unsigned*>(in)[i];
    I = (short)(w & 0xffffu);
    Q = (short)(w >> 16);
  }
  else
  {
    const unsigned w = reinterpret_cast<const unsigned short*>(in)[i];
    I = F == kIqS8 ? (int)(signed char)(w & 0xffu) : (int)(w & 0xffu);
    Q = F == kIqS8 ? (int)(signed char)(w >> 8) : (int)(w >> 8);
  }
}

template <int F>
__global__ void __launch_bounds__(kStThreads) k_iq_stats(const void* __restrict__ in, uint64_t n,
                                                         typename StAcc<F>::T* __restrict__ partial)
{
  using T = typename StAcc<F>::T;
  __shared__ T warp_sum[kStThreads / 32][kStSums];
  const unsigned tid = threadIdx.x;
  const uint64_t base = (uint64_t)blockIdx.x * kStChunk + tid;
  T s[kStSums] = {0, 0, 0, 0, 0};
#pragma unroll 8
  for (unsigned j = 0; j < kStPerThread; ++j)
  {
    const uint64_t i = base + (uint64_t)j * kStThreads;
    if (i < n)
    {
      if constexpr (F == kIqCF32)
      {
        const float2 v = reinterpret_cast<const float2*>(in)[i];
        const double I = v.x, Q = v.y;
        s[0] = s[0] + I;
        s[1] = s[1] + Q;
        s[2] = s[2] + I * I;
        s[3] = s[3] + Q * Q;
        s[4] = s[4] + I * Q;
      }
      else
      {
        int I, Q;
        st_codes<F>(in, i, I, Q);
        s[0] += I;
        s[1] += Q;
        s[2] += (long long)(I * I);
        s[3] += (long long)(Q * Q);
        s[4] += (long long)(I * Q);
      }
    }
  }
#pragma unroll
  for (unsigned k = 0; k < kStSums; ++k)
  {
#pragma unroll
    for (unsigned o = 16; o > 0; o >>= 1)
      s[k] = s[k] + __shfl_xor_sync(0xffffffffu, s[k], o);
  }
  if ((tid & 31u) == 0)
    for (unsigned k = 0; k < kStSums; ++k)
      warp_sum[tid >> 5][k] = s[k];
  __syncthreads();
  if (tid < kStSums)
  {
    T acc = warp_sum[0][tid];
    for (unsigned w = 1; w < kStThreads / 32; ++w)
      acc = acc + warp_sum[w][tid];
    partial[(size_t)blockIdx.x * kStSums + tid] = acc;
  }
}

template <typename T>
__global__ void __launch_bounds__(kStThreads) k_iq_stats_reduce(const T* __restrict__ partial, unsigned rows,
                                                                T* __restrict__ out)
{
  __shared__ T part[kStSums][kStThreads];
  const unsigned tid = threadIdx.x;
  T s[kStSums] = {0, 0, 0, 0, 0};
  for (unsigned r = tid; r < rows; r += kStThreads)
#pragma unroll
    for (unsigned k = 0; k < kStSums; ++k)
      s[k] = s[k] + partial[(size_t)r * kStSums + k];
#pragma unroll
  for (unsigned k = 0; k < kStSums; ++k)
    part[k][tid] = s[k];
  __syncthreads();
  if (tid < kStSums)
  {
    T acc = part[tid][0];
    for (unsigned t = 1; t < kStThreads; ++t)
      acc = acc + part[tid][t];
    out[tid] = acc;
  }
}

int EstFail(int code, const std::string& m)
{
  rfm::SetLastError(m);
  return code;
}

// a, b from the moments (the same expressions as oracle/iqcorr.py)
void Imbalance(double vI, double vQ, double c, rfm_iq_correction* out)
{
  double a = 1.0, b = 0.0;
  bool ok = vI > 0.0 && vI * vQ - c * c > 0.0;
  if (ok)
  {
    a = sqrt(vI / (vQ - c * c / vI));
    b = -a * c / vI;
    ok = isfinite(a) && isfinite(b);
  }
  out->a = ok ? (float)a : 1.0f;
  out->b = ok ? (float)b : 0.0f;
  out->imbalance_valid = ok ? 1 : 0;
}

void IqCoefficientsInt(int fmt, uint64_t n, const long long* S, rfm_iq_correction* out)
{
  const __int128 N = (__int128)n;
  const __int128 vi = N * S[2] - (__int128)S[0] * S[0];
  const __int128 vq = N * S[3] - (__int128)S[1] * S[1];
  const __int128 cc = N * S[4] - (__int128)S[0] * S[1];
  const double nn = (double)n;
  const double k = fmt == kIqU8 ? 1.0 / 127.5 : (fmt == kIqS8 ? 0x1p-7 : 0x1p-15);
  const double k2 = k * k, n2 = nn * nn;
  if (fmt == kIqU8)
  {
    out->dc_i = (float)((double)S[0] / nn / 127.5 - 1.0);
    out->dc_q = (float)((double)S[1] / nn / 127.5 - 1.0);
  }
  else
  {
    out->dc_i = (float)((double)S[0] / nn * k);
    out->dc_q = (float)((double)S[1] / nn * k);
  }
  Imbalance((double)vi / n2 * k2, (double)vq / n2 * k2, (double)cc / n2 * k2, out);
}

void IqCoefficientsF64(uint64_t n, const double* S, rfm_iq_correction* out)
{
  const double nn = (double)n;
  const double mi = S[0] / nn, mq = S[1] / nn;
  out->dc_i = (float)mi;
  out->dc_q = (float)mq;
  Imbalance(S[2] / nn - mi * mi, S[3] / nn - mq * mq, S[4] / nn - mi * mq, out);
}
} // namespace

namespace rfm
{
// The estimate of n samples of format fmt at device pointer d_in (validated by the caller), on stream st; blocking.
int IqEstimateDevice(int fmt, const void* d_in, uint64_t n, cudaStream_t st, rfm_iq_correction* out)
{
  const uint64_t rows = (n + kStChunk - 1) / kStChunk;
  void* scratch = nullptr;
  if (cudaMalloc(&scratch, (size_t)(rows + 1) * kStSums * 8) != cudaSuccess)
    return EstFail(RFM_ERR_CUDA, "rfm_iq_estimate: scratch allocation failed");
  unsigned long long sums[kStSums] = {0, 0, 0, 0, 0};
#define RFM_IQ_STATS(F, T)                                                                                             \
  {                                                                                                                    \
    T* part = static_cast<T*>(scratch);                                                                                \
    k_iq_stats<F><<<(unsigned)rows, kStThreads, 0, st>>>(d_in, n, part);                                               \
    k_iq_stats_reduce<T><<<1, kStThreads, 0, st>>>(part, (unsigned)rows, part + rows * kStSums);                       \
  }
  switch (fmt)
  {
    case kIqU8: RFM_IQ_STATS(kIqU8, long long); break;
    case kIqS8: RFM_IQ_STATS(kIqS8, long long); break;
    case kIqS16: RFM_IQ_STATS(kIqS16, long long); break;
    default: RFM_IQ_STATS(kIqCF32, double); break;
  }
#undef RFM_IQ_STATS
  g_launches += 2;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(sums, static_cast<unsigned long long*>(scratch) + rows * kStSums, sizeof(sums),
                        cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess)
    e = cudaStreamSynchronize(st);
  cudaFree(scratch);
  if (e != cudaSuccess)
    return EstFail(RFM_ERR_CUDA, std::string("rfm_iq_estimate: statistics pass failed: ") + cudaGetErrorString(e));
  if (fmt == kIqCF32)
    IqCoefficientsF64(n, reinterpret_cast<const double*>(sums), out);
  else
    IqCoefficientsInt(fmt, n, reinterpret_cast<const long long*>(sums), out);
  return RFM_OK;
}

// the checks every entry point applies to a capture it estimates from
int IqEstimateCheck(const char* who, int fmt, const void* iq, uint64_t n, bool on_device)
{
  const uint32_t esz = rfm_iq_format_bytes(fmt);
  if (esz == 0)
    return EstFail(RFM_ERR_INVALID, std::string(who) + ": unknown IQ format");
  if (!iq || n == 0)
    return EstFail(RFM_ERR_INVALID, std::string(who) + ": empty capture");
  if (n > (1ull << 32))
    return EstFail(RFM_ERR_INVALID, std::string(who) + ": more than 2^32 samples (the integer statistics' limit)");
  if (on_device && reinterpret_cast<uintptr_t>(iq) % esz != 0)
    return EstFail(RFM_ERR_INVALID, std::string(who) + ": device capture must be aligned to the sample size "
                                                       "(2 / 2 / 4 / 8 bytes for u8 / s8 / s16 / cf32)");
  return RFM_OK;
}
} // namespace rfm

extern "C"
{

int rfm_iq_estimate(int format, const void* iq, uint64_t n, int iq_on_device, int device, rfm_iq_correction* out)
{
  if (!out)
    return EstFail(RFM_ERR_INVALID, "rfm_iq_estimate: null output");
  int rc = rfm::IqEstimateCheck("rfm_iq_estimate", format, iq, n, iq_on_device != 0);
  if (rc != RFM_OK)
    return rc;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return EstFail(RFM_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
  if (device < 0 && cudaGetDevice(&device) != cudaSuccess)
    return EstFail(RFM_ERR_CUDA, "cudaGetDevice failed");
  if (device >= ndev || cudaSetDevice(device) != cudaSuccess)
    return EstFail(RFM_ERR_INVALID, "rfm_iq_estimate: device ordinal out of range");
  const void* d_in = iq;
  void* staging = nullptr;
  if (!iq_on_device)
  {
    const size_t bytes = (size_t)n * rfm_iq_format_bytes(format);
    if (cudaMalloc(&staging, bytes) != cudaSuccess)
      return EstFail(RFM_ERR_CUDA, "rfm_iq_estimate: capture allocation failed");
    if (cudaMemcpy(staging, iq, bytes, cudaMemcpyHostToDevice) != cudaSuccess)
    {
      cudaFree(staging);
      return EstFail(RFM_ERR_CUDA, "rfm_iq_estimate: H2D copy failed");
    }
    d_in = staging;
  }
  rc = rfm::IqEstimateDevice(format, d_in, n, 0, out);
  cudaFree(staging);
  return rc;
}

} // extern "C"
