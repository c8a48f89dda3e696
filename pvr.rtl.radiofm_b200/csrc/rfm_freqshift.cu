// rfm_freqshift.cu -- cFreqShift (FreqShift.h:12-27, FreqShift.cpp:10-76) on the GPU, batched over rows (one row per
// station of a wideband capture, or per stream), optionally fused with the u8 -> float conversion of
// cRtlSdrSource::ReadAsyncCB (RTL_SDR_Source.cpp:207-211) or the exact s8 / s16 -> float conversions (rfm_dsp.cuh).
//
// Bug-compatible with the reference's x86 branch: the NCO phase is a float32 that is advanced by a float32 increment
// and NEVER wrapped (FreqShift.cpp:71-72).  The phase sequence is therefore a sequential float recurrence
// (phase = fl(phase + inc)); it is produced by one lane per row (k_fs_phase, 1 dependent FADD per sample) and the
// mixing itself -- sin/cos of the phase (== x87 fsincos rounded to float, rfm_math.cuh), complex multiply with
// individually rounded products (4 mul, 2 add) -- runs fully parallel (k_fs_mix).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/radiofm_b200.h"
#include "rfm_dsp.cuh"
#include "rfm_math.cuh"

using namespace rfm;

namespace rfm
{
void SetLastError(const std::string& m);
}

namespace
{
__global__ void __launch_bounds__(32) k_fs_phase(const float* inc, float* time, float* ph, size_t ph_stride, unsigned n,
                                                 unsigned rows)
{
  __shared__ float tile[32][33];
  const unsigned lane = threadIdx.x;
  const unsigned r0 = blockIdx.x * 32, r = r0 + lane;
  const bool valid = r < rows;
  float acc = valid ? time[r] : 0.0f;
  const float step = valid ? inc[r] : 0.0f;
  for (unsigned t0 = 0; t0 < n; t0 += 32)
  {
    const unsigned tn = min(32u, n - t0);
    for (unsigned k = 0; k < tn; ++k)
    {
      tile[lane][k] = acc;             // phase used for sample t0 + k (FreqShift.cpp:55-56)
      acc = addf(acc, step);           // :71 m_NcoTime += m_NcoInc
    }
    __syncwarp();
    if (lane < tn)
      for (unsigned q = 0; q < 32 && r0 + q < rows; ++q)
        ph[(size_t)(r0 + q) * ph_stride + t0 + lane] = tile[q][lane];
    __syncwarp();
  }
  if (valid)
    time[r] = acc;
}

// F: IqFormat of the input rows (cf32 rows may be mixed in place), or of one capture shared by every row (SHARED; a
// shared cf32 capture is read as rows of stride 0).  CORR: the IQ correction follows the conversion (rfm_iq_correct).
template <int F, bool SHARED, bool CORR>
__global__ void __launch_bounds__(256) k_fs_mix(const float* ph, size_t ph_stride, const void* in, size_t in_stride,
                                                float2* out, size_t out_stride, unsigned n, const float* lut, IqCorr corr)
{
  const unsigned i = blockIdx.x * 256 + threadIdx.x;
  const unsigned r = blockIdx.y;
  if (i >= n)
    return;
  float s, c;
  rfm_sincos(ph[(size_t)r * ph_stride + i], &s, &c);
  float2 d;
  if (F == kIqCF32)
    d = reinterpret_cast<const float2*>(in)[(size_t)r * in_stride + i];
  else if (F == kIqU8)
  {
    const uchar2 u = reinterpret_cast<const uchar2*>(in)[(SHARED ? 0 : (size_t)r * in_stride) + i];
    d = make_float2(lut[u.x], lut[u.y]);
  }
  else if (F == kIqS8)
  {
    const unsigned w = reinterpret_cast<const unsigned short*>(in)[(SHARED ? 0 : (size_t)r * in_stride) + i];
    d = make_float2(rfm_s8_to_float(w, 0u), rfm_s8_to_float(w, 1u));
  }
  else
  {
    const unsigned w = reinterpret_cast<const unsigned*>(in)[(SHARED ? 0 : (size_t)r * in_stride) + i];
    d = make_float2(rfm_s16_to_float(w, 0u), rfm_s16_to_float(w, 1u));
  }
  if (CORR)
    d = rfm_iq_correct(d, corr);
  float2 o;
  o.x = subf(mulf(d.x, c), mulf(d.y, s)); // FreqShift.cpp:63-69
  o.y = addf(mulf(d.x, s), mulf(d.y, c));
  out[(size_t)r * out_stride + i] = o;
}
} // namespace

struct rfm_freqshift
{
  unsigned rows = 0, cap = 0;
  int device = 0;
  float *d_inc = nullptr, *d_time = nullptr, *d_ph = nullptr, *d_lut = nullptr, *d_time_end = nullptr;
  // Reset() before every block (phase-coherent blocks of a wideband capture) repeats the same phase sequence: the
  // table computed from phase 0 is kept and the sequential k_fs_phase pass skipped when the next call is identical
  bool at_zero = true;
  unsigned ph0_n = 0;
  float2* d_io = nullptr;
  uint8_t* d_raw = nullptr;   // host input of the _iq / _u8 calls, raw_bytes
  size_t raw_bytes = 0;
  std::string err;
  bool corr_on = false;      // rfm_freqshift_set_iq_correction
  IqCorr corr = {0.f, 0.f, 1.f, 0.f};
};

extern "C"
{

int rfm_freqshift_create(uint32_t rows, const float* nco_freq, float in_rate, uint32_t max_len, int device,
                         rfm_freqshift** out)
{
  if (!out || !nco_freq || rows == 0 || max_len == 0 || !(in_rate > 0))
    return RFM_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return RFM_ERR_NO_DEVICE;
  if (device < 0)
    cudaGetDevice(&device);
  if (cudaSetDevice(device) != cudaSuccess)
    return RFM_ERR_CUDA;
  rfm_freqshift* f = new rfm_freqshift;
  f->rows = rows; f->cap = max_len; f->device = device;
  std::vector<float> inc(rows), lut(256);
  for (uint32_t r = 0; r < rows; ++r)
    inc[r] = (float)((2.0 * 3.14159265358979323846) * nco_freq[r] / in_rate); // FreqShift.cpp:15 (K_2PI is double)
  for (int u = 0; u < 256; ++u)
    lut[u] = (float)(u / (255.0 / 2.0) - 1.0);
  bool ok = cudaMalloc(&f->d_inc, rows * 4) == cudaSuccess && cudaMalloc(&f->d_time, rows * 4) == cudaSuccess &&
            cudaMalloc(&f->d_ph, (size_t)rows * max_len * 4) == cudaSuccess && cudaMalloc(&f->d_lut, 1024) == cudaSuccess &&
            cudaMalloc(&f->d_time_end, rows * 4) == cudaSuccess &&
            cudaMalloc(&f->d_io, (size_t)rows * max_len * 8) == cudaSuccess &&
            cudaMalloc(&f->d_raw, (size_t)rows * max_len * 2) == cudaSuccess;
  f->raw_bytes = ok ? (size_t)rows * max_len * 2 : 0;
  if (ok)
  {
    cudaMemcpy(f->d_inc, inc.data(), rows * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(f->d_lut, lut.data(), 1024, cudaMemcpyHostToDevice);
    ok = cudaMemset(f->d_time, 0, rows * 4) == cudaSuccess;
  }
  if (!ok)
  {
    rfm_freqshift_destroy(f);
    return RFM_ERR_CUDA;
  }
  *out = f;
  return RFM_OK;
}

void rfm_freqshift_destroy(rfm_freqshift* f)
{
  if (!f)
    return;
  cudaSetDevice(f->device);
  cudaFree(f->d_time_end);
  cudaFree(f->d_inc); cudaFree(f->d_time); cudaFree(f->d_ph); cudaFree(f->d_lut); cudaFree(f->d_io); cudaFree(f->d_raw);
  delete f;
}

int rfm_freqshift_reset(rfm_freqshift* f) // FreqShift.cpp:18-21
{
  if (!f)
    return RFM_ERR_INVALID;
  cudaSetDevice(f->device);
  f->at_zero = true;
  return cudaMemsetAsync(f->d_time, 0, f->rows * 4, 0) == cudaSuccess ? RFM_OK : RFM_ERR_CUDA;
}

static int Run(rfm_freqshift* f, int fmt, bool shared, const void* d_in, size_t in_stride, float2* d_out,
               size_t out_stride, uint32_t n, cudaStream_t st)
{
  if (f->at_zero && f->ph0_n == n)
    cudaMemcpyAsync(f->d_time, f->d_time_end, f->rows * 4, cudaMemcpyDeviceToDevice, st); // table still valid
  else
  {
    k_fs_phase<<<(f->rows + 31) / 32, 32, 0, st>>>(f->d_inc, f->d_time, f->d_ph, f->cap, n, f->rows);
    f->ph0_n = 0;
    if (f->at_zero)
    {
      cudaMemcpyAsync(f->d_time_end, f->d_time, f->rows * 4, cudaMemcpyDeviceToDevice, st);
      f->ph0_n = n;
    }
  }
  f->at_zero = false;
  dim3 grid((n + 255) / 256, f->rows);
#define RFM_FS_MIX(F, SHARED)                                                                                          \
  if (f->corr_on)                                                                                                      \
    k_fs_mix<F, SHARED, true><<<grid, 256, 0, st>>>(f->d_ph, f->cap, d_in, in_stride, d_out, out_stride, n, f->d_lut,   \
                                                    f->corr);                                                          \
  else                                                                                                                 \
    k_fs_mix<F, SHARED, false><<<grid, 256, 0, st>>>(f->d_ph, f->cap, d_in, in_stride, d_out, out_stride, n, f->d_lut,  \
                                                     f->corr)
  switch (fmt)
  {
    case kIqU8: if (shared) { RFM_FS_MIX(kIqU8, true); } else { RFM_FS_MIX(kIqU8, false); } break;
    case kIqS8: if (shared) { RFM_FS_MIX(kIqS8, true); } else { RFM_FS_MIX(kIqS8, false); } break;
    case kIqS16: if (shared) { RFM_FS_MIX(kIqS16, true); } else { RFM_FS_MIX(kIqS16, false); } break;
    default: in_stride = shared ? 0 : in_stride; RFM_FS_MIX(kIqCF32, false); break;
  }
#undef RFM_FS_MIX
  return cudaGetLastError() == cudaSuccess ? RFM_OK : RFM_ERR_CUDA;
}

int rfm_freqshift_set_iq_correction(rfm_freqshift* f, const rfm_iq_correction* c)
{
  if (!f)
    return RFM_ERR_INVALID;
  if (c && !(isfinite(c->dc_i) && isfinite(c->dc_q) && isfinite(c->a) && isfinite(c->b)))
  {
    rfm::SetLastError("rfm_freqshift_set_iq_correction: coefficients must be finite");
    return RFM_ERR_INVALID;
  }
  f->corr_on = c != nullptr;
  f->corr = c ? IqCorr{c->dc_i, c->dc_q, c->a, c->b} : IqCorr{0.f, 0.f, 1.f, 0.f};
  return RFM_OK;
}

int rfm_freqshift_process_cf32(rfm_freqshift* f, float* iq, uint32_t n)
{
  if (!f || !iq || n > f->cap)
    return RFM_ERR_INVALID;
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  const size_t bytes = (size_t)f->rows * n * 8;
  if (cudaMemcpy(f->d_io, iq, bytes, cudaMemcpyHostToDevice) != cudaSuccess)
    return RFM_ERR_CUDA;
  int rc = Run(f, kIqCF32, false, f->d_io, n, f->d_io, n, n, 0);
  if (rc == RFM_OK && cudaMemcpy(iq, f->d_io, bytes, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = RFM_ERR_CUDA;
  return rc;
}

int rfm_freqshift_process_iq(rfm_freqshift* f, int format, int shared_capture, const void* iq, uint32_t n, float* out)
{
  const uint32_t esz = rfm_iq_format_bytes(format);
  if (!f || !iq || !out || n > f->cap || esz == 0)
    return RFM_ERR_INVALID;
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  const size_t in_bytes = (size_t)(shared_capture ? 1 : f->rows) * n * esz;
  if (f->raw_bytes < in_bytes)
  {
    cudaFree(f->d_raw);
    f->d_raw = nullptr;
    f->raw_bytes = 0;
    if (cudaMalloc(&f->d_raw, in_bytes) != cudaSuccess)
      return RFM_ERR_CUDA;
    f->raw_bytes = in_bytes;
  }
  if (cudaMemcpyAsync(f->d_raw, iq, in_bytes, cudaMemcpyHostToDevice, 0) != cudaSuccess)
    return RFM_ERR_CUDA;
  int rc = Run(f, format, shared_capture != 0, f->d_raw, n, f->d_io, n, n, 0);
  if (rc == RFM_OK && (cudaMemcpyAsync(out, f->d_io, (size_t)f->rows * n * 8, cudaMemcpyDeviceToHost, 0) != cudaSuccess ||
                       cudaStreamSynchronize(0) != cudaSuccess))
    rc = RFM_ERR_CUDA;
  return rc;
}

int rfm_freqshift_process_u8(rfm_freqshift* f, const uint8_t* iq, int shared_capture, uint32_t n, float* out)
{
  return rfm_freqshift_process_iq(f, RFM_IQ_U8, shared_capture, iq, n, out);
}

int rfm_freqshift_process_iq_device(rfm_freqshift* f, int format, int shared_capture, const void* d_in, size_t in_stride,
                                    float* d_out, size_t out_stride, uint32_t n, void* cuda_stream)
{
  const uint32_t esz = rfm_iq_format_bytes(format);
  if (!f || !d_in || !d_out || n > f->cap || esz == 0)
    return RFM_ERR_INVALID;
  if (reinterpret_cast<uintptr_t>(d_in) % esz != 0)
  {
    rfm::SetLastError("rfm_freqshift_process_iq_device: d_in must be aligned to the sample size (2 / 2 / 4 / 8 bytes for "
                      "u8 / s8 / s16 / cf32)");
    return RFM_ERR_INVALID;
  }
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  return Run(f, format, shared_capture != 0, d_in, in_stride, reinterpret_cast<float2*>(d_out), out_stride, n,
             static_cast<cudaStream_t>(cuda_stream));
}

int rfm_freqshift_process_device(rfm_freqshift* f, int mode, const void* d_in, size_t in_stride, float* d_out,
                                 size_t out_stride, uint32_t n, void* cuda_stream)
{
  if (!f || !d_in || !d_out || n > f->cap || mode < 0 || mode > 2)
    return RFM_ERR_INVALID;
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  return Run(f, mode == 0 ? kIqCF32 : kIqU8, mode == 1, d_in, in_stride, reinterpret_cast<float2*>(d_out), out_stride, n,
             static_cast<cudaStream_t>(cuda_stream));
}

} // extern "C"
