// rfm_primitives.cu -- the reference's filter classes as stand-alone batched GPU primitives behind the C ABI, so that
// the drop-in host classes (pvr.rtl.radiofm_b200/host/*.h) are one-line forwards:
//
//   rfm_iir      cIirFilter            (IirFilter.h:12-36, IirFilter.cpp:11-105): RBJ biquad LP/HP/BP/BR, DF-II
//   rfm_fir      cFirFilter            (FirFilter.h:17-60, FirFilter.cpp:78-148,195-264,273-413): Kaiser LP / HP design / constant taps,
//                                      circular delay line with its rotating summation start
//   rfm_rdsproc  cRDSRxSignalProcessor (RDSProcess.h:56-110, RDSProcess.cpp:43-180): 57 kHz mix, decimation, LP, Costas
//                                      loop, matched filter, bit clock / slicer on the device; block sync + FEC on the
//                                      host (rfm_rdssync)
//
// One row per independent stream.  The kernels are the ones of the fused chain (k_rotfir, k_rds_front, k_rds_pll,
// k_rds_slice, ... in rfm_kernels.cu) plus a lane-per-row biquad; the arithmetic is the reference's, operation by
// operation (rfm_math.cuh), so every primitive is bit-exact against the oracle on its own.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <string>
#include <vector>

#include "../../include/radiofm_b200.h"
#include "rfm_dsp.cuh"
#include "rfm_kernels.cuh"
#include "rfm_plan.h"
#include "rfm_rdssync.h"

using namespace rfm;

namespace rfm
{
extern std::atomic<uint64_t> g_launches;
void SetLastError(const std::string& m);
}

namespace
{
int PFail(int code, const std::string& m)
{
  rfm::SetLastError(m);
  return code;
}

template <typename T>
bool DevAllocZ(T** p, size_t n)
{
  const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
  return cudaMalloc(reinterpret_cast<void**>(p), bytes) == cudaSuccess && cudaMemset(*p, 0, bytes) == cudaSuccess;
}

int PickDevice(int* device)
{
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return PFail(RFM_ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)");
  if (*device < 0)
    cudaGetDevice(device);
  if (cudaSetDevice(*device) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "cudaSetDevice failed");
  return RFM_OK;
}

// --------------------------------------------------------------------------------------------------
// cIirFilter::Process / ProcessTwo, IirFilter.cpp:62-105.  A warp owns 32 rows and walks them in tiles of 32 samples:
// coalesced row accesses into a shared tile, each lane then runs its row's recurrence down a tile column.
// MODE 0: real rows; 1: complex rows (re and im are two independent filters, :62-76); 2: two real buffers (:89-105)
// --------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(32) k_iir(BiquadDev c, float* a, float* b, size_t stride, unsigned n, unsigned rows,
                                            float* state)
{
  constexpr int CH = MODE == 0 ? 1 : 2;
  __shared__ float tile[CH][32][33];
  const unsigned lane = threadIdx.x;
  const unsigned r0 = blockIdx.x * 32, r = r0 + lane;
  const bool valid = r < rows;
  float w1a = 0.f, w2a = 0.f, w1b = 0.f, w2b = 0.f;
  if (valid)
  {
    w1a = state[0 * rows + r]; w2a = state[1 * rows + r];
    w1b = state[2 * rows + r]; w2b = state[3 * rows + r];
  }
  for (unsigned t0 = 0; t0 < n; t0 += 32)
  {
    const unsigned tn = min(32u, n - t0);
    for (unsigned q = 0; q < 32 && r0 + q < rows; ++q)
    {
      if (MODE == 1)
      {
        // interleaved re, im: 64 floats per row tile
        const float* src = a + ((size_t)(r0 + q) * stride + t0) * 2;
        if (lane < tn) { tile[0][q][lane] = src[2 * lane]; tile[1][q][lane] = src[2 * lane + 1]; }
      }
      else
      {
        if (lane < tn)
        {
          tile[0][q][lane] = a[(size_t)(r0 + q) * stride + t0 + lane];
          if (MODE == 2) tile[1][q][lane] = b[(size_t)(r0 + q) * stride + t0 + lane];
        }
      }
    }
    __syncwarp();
    if (valid)
      for (unsigned k = 0; k < tn; ++k)
      {
        tile[0][lane][k] = biquad_step(c, tile[0][lane][k], w1a, w2a);
        if (CH == 2) tile[1][lane][k] = biquad_step(c, tile[1][lane][k], w1b, w2b);
      }
    __syncwarp();
    for (unsigned q = 0; q < 32 && r0 + q < rows; ++q)
    {
      if (MODE == 1)
      {
        float* dst = a + ((size_t)(r0 + q) * stride + t0) * 2;
        if (lane < tn) { dst[2 * lane] = tile[0][q][lane]; dst[2 * lane + 1] = tile[1][q][lane]; }
      }
      else if (lane < tn)
      {
        a[(size_t)(r0 + q) * stride + t0 + lane] = tile[0][q][lane];
        if (MODE == 2) b[(size_t)(r0 + q) * stride + t0 + lane] = tile[1][q][lane];
      }
    }
    __syncwarp();
  }
  if (valid)
  {
    state[0 * rows + r] = w1a; state[1 * rows + r] = w2a;
    state[2 * rows + r] = w1b; state[3 * rows + r] = w2b;
  }
}

// copy rows [rows][n] (elem bytes each) into V rows at element offset `hist`
__global__ void __launch_bounds__(256) k_to_v(const char* src, size_t src_stride_b, char* dst, size_t dst_stride_b,
                                              unsigned hist, unsigned n, unsigned elem)
{
  const unsigned i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n)
    return;
  const char* s = src + (size_t)blockIdx.y * src_stride_b + (size_t)i * elem;
  char* d = dst + (size_t)blockIdx.y * dst_stride_b + (size_t)(hist + i) * elem;
  if (elem == 4)
    *reinterpret_cast<float*>(d) = *reinterpret_cast<const float*>(s);
  else
    *reinterpret_cast<float2*>(d) = *reinterpret_cast<const float2*>(s);
}
// (a, b) real rows -> complex V rows at element offset `hist` (ProcessTwo stores ComplexType(bufferA[i], bufferB[i]) in the
// complex delay line, FirFilter.cpp:397), and back
__global__ void __launch_bounds__(256) k_join_v(const float* a, const float* b, size_t stride, float2* v, size_t v_stride,
                                                unsigned hist, unsigned n)
{
  const unsigned i = blockIdx.x * 256 + threadIdx.x;
  if (i < n)
    v[(size_t)blockIdx.y * v_stride + hist + i] = make_float2(a[(size_t)blockIdx.y * stride + i], b[(size_t)blockIdx.y * stride + i]);
}

__global__ void __launch_bounds__(256) k_split(const float2* t, size_t t_stride, float* a, float* b, size_t stride, unsigned n)
{
  const unsigned i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n)
    return;
  const float2 v = t[(size_t)blockIdx.y * t_stride + i];
  a[(size_t)blockIdx.y * stride + i] = v.x;
  b[(size_t)blockIdx.y * stride + i] = v.y;
}
} // namespace

// ==================================================================================================
// cIirFilter
// ==================================================================================================
struct rfm_iir
{
  unsigned rows = 0, cap = 0;
  int device = 0;
  Biquad c{0, 0, 0, 0, 0};
  bool inited = false;
  float *d_state = nullptr, *d_a = nullptr, *d_b = nullptr;
};

extern "C"
{

int rfm_iir_create(uint32_t rows, uint32_t max_len, int device, rfm_iir** out)
{
  if (!out || rows == 0 || max_len == 0)
    return PFail(RFM_ERR_INVALID, "rfm_iir_create: invalid argument");
  *out = nullptr;
  int rc = PickDevice(&device);
  if (rc != RFM_OK)
    return rc;
  rfm_iir* f = new rfm_iir;
  f->rows = rows; f->cap = max_len; f->device = device;
  if (!DevAllocZ(&f->d_state, 4 * (size_t)rows))
  {
    rfm_iir_destroy(f);
    return PFail(RFM_ERR_CUDA, "rfm_iir_create: device allocation failed");
  }
  *out = f;
  return RFM_OK;
}

void rfm_iir_destroy(rfm_iir* f)
{
  if (!f)
    return;
  cudaSetDevice(f->device);
  cudaFree(f->d_state); cudaFree(f->d_a); cudaFree(f->d_b);
  delete f;
}

// cIirFilter::Init, IirFilter.cpp:11-60: coefficients + cleared delays.  Unknown type: the reference returns false after
// clearing the delays and leaves the old coefficients; so does this (RFM_ERR_INVALID).
int rfm_iir_init(rfm_iir* f, int type, float F0, float Q, float Fs)
{
  if (!f)
    return PFail(RFM_ERR_INVALID, "rfm_iir_init: null handle");
  cudaSetDevice(f->device);
  Biquad c;
  const bool ok = PlanBiquad(type, F0, Q, Fs, &c);
  if (ok)
  {
    f->c = c;
    f->inited = true;
  }
  if (cudaMemsetAsync(f->d_state, 0, 4 * (size_t)f->rows * sizeof(float), 0) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_iir_init: state reset failed");
  return ok ? RFM_OK : PFail(RFM_ERR_INVALID, "rfm_iir_init: unknown filter type (cIirFilter::Init returns false)");
}

int rfm_iir_coefficients(const rfm_iir* f, float* out5)
{
  if (!f || !out5)
    return PFail(RFM_ERR_INVALID, "rfm_iir_coefficients: invalid argument");
  out5[0] = f->c.A1; out5[1] = f->c.A2; out5[2] = f->c.B0; out5[3] = f->c.B1; out5[4] = f->c.B2;
  return RFM_OK;
}

int rfm_iir_process_device(rfm_iir* f, int mode, float* d_a, float* d_b, size_t stride, uint32_t n, void* cuda_stream)
{
  if (!f || !d_a || mode < 0 || mode > 2 || (mode == 2 && !d_b))
    return PFail(RFM_ERR_INVALID, "rfm_iir_process_device: invalid argument");
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  const BiquadDev c{f->c.A1, f->c.A2, f->c.B0, f->c.B1, f->c.B2};
  const unsigned grid = (f->rows + 31) / 32;
  if (mode == 0)
    k_iir<0><<<grid, 32, 0, st>>>(c, d_a, nullptr, stride, n, f->rows, f->d_state);
  else if (mode == 1)
    k_iir<1><<<grid, 32, 0, st>>>(c, d_a, nullptr, stride, n, f->rows, f->d_state);
  else
    k_iir<2><<<grid, 32, 0, st>>>(c, d_a, d_b, stride, n, f->rows, f->d_state);
  ++rfm::g_launches;
  return cudaGetLastError() == cudaSuccess ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_iir: kernel launch failed");
}

static int IirHost(rfm_iir* f, int mode, float* a, float* b, uint32_t n)
{
  if (!f || !a || (mode == 2 && !b) || n > f->cap)
    return PFail(RFM_ERR_INVALID, "rfm_iir_process: invalid argument");
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  const size_t elems = (size_t)f->rows * f->cap * 2;
  if (!f->d_a && !DevAllocZ(&f->d_a, elems))
    return PFail(RFM_ERR_CUDA, "rfm_iir: staging allocation failed");
  if (mode == 2 && !f->d_b && !DevAllocZ(&f->d_b, elems))
    return PFail(RFM_ERR_CUDA, "rfm_iir: staging allocation failed");
  const size_t bytes = (size_t)f->rows * n * (mode == 1 ? 8 : 4);
  if (cudaMemcpy(f->d_a, a, bytes, cudaMemcpyHostToDevice) != cudaSuccess ||
      (mode == 2 && cudaMemcpy(f->d_b, b, bytes, cudaMemcpyHostToDevice) != cudaSuccess))
    return PFail(RFM_ERR_CUDA, "rfm_iir: H2D copy failed");
  int rc = rfm_iir_process_device(f, mode, f->d_a, f->d_b, n, n, nullptr);
  if (rc != RFM_OK)
    return rc;
  if (cudaMemcpy(a, f->d_a, bytes, cudaMemcpyDeviceToHost) != cudaSuccess ||
      (mode == 2 && cudaMemcpy(b, f->d_b, bytes, cudaMemcpyDeviceToHost) != cudaSuccess))
    return PFail(RFM_ERR_CUDA, "rfm_iir: D2H copy failed");
  return RFM_OK;
}

int rfm_iir_process_real(rfm_iir* f, float* buf, uint32_t n) { return IirHost(f, 0, buf, nullptr, n); }
int rfm_iir_process_complex(rfm_iir* f, float* buf, uint32_t n) { return IirHost(f, 1, buf, nullptr, n); }
int rfm_iir_process_two(rfm_iir* f, float* a, float* b, uint32_t n) { return IirHost(f, 2, a, b, n); }

} // extern "C"

// ==================================================================================================
// cFirFilter
// ==================================================================================================
struct rfm_fir
{
  unsigned rows = 0, cap = 0, taps = 0, g = 0; // g: samples filtered since the last Init, mod taps (m_State)
  int device = 0;
  std::vector<float> coef;
  float* d_coef = nullptr;
  // V rows [rows][v_stride] of cf32-sized slots: d_va = m_rZBuf (real Process), d_vb = m_cZBuf (complex Process AND
  // ProcessTwo, which keeps (A, B) as (re, im) in the same delay line: FirFilter.cpp:337,397)
  float *d_va = nullptr, *d_vb = nullptr;
  float2* d_tmp = nullptr;                // ProcessTwo: complex result before it is split into A and B
  size_t v_stride = 0;
  float *d_a = nullptr, *d_b = nullptr;   // staging for the host entry points
};

namespace
{
int FirInstall(rfm_fir* f, const std::vector<float>& taps)
{
  if (taps.empty() || taps.size() > kMaxFirTaps)
    return PFail(RFM_ERR_UNSUPPORTED, "rfm_fir: tap count outside 1..75 (cFirFilter MAX_NUMCOEF, FirFilter.h:15)");
  f->coef = taps;
  f->taps = (unsigned)taps.size();
  f->g = 0; // FirFilter.cpp:145,319
  const size_t vbytes = (size_t)f->rows * f->v_stride * sizeof(float2);
  if (cudaMemcpy(f->d_coef, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemset(f->d_va, 0, vbytes) != cudaSuccess || cudaMemset(f->d_vb, 0, vbytes) != cudaSuccess) // :138-144,313-319
    return PFail(RFM_ERR_CUDA, "rfm_fir: upload failed");
  return RFM_OK;
}
} // namespace

extern "C"
{

int rfm_fir_create(uint32_t rows, uint32_t max_len, int device, rfm_fir** out)
{
  if (!out || rows == 0 || max_len == 0)
    return PFail(RFM_ERR_INVALID, "rfm_fir_create: invalid argument");
  *out = nullptr;
  int rc = PickDevice(&device);
  if (rc != RFM_OK)
    return rc;
  rfm_fir* f = new rfm_fir;
  f->rows = rows; f->cap = max_len; f->device = device;
  f->v_stride = ((size_t)kMaxFirTaps + max_len + 15) & ~(size_t)15;
  float2 *va = nullptr, *vb = nullptr;
  const bool ok = DevAllocZ(&f->d_coef, kMaxFirTapsDev) && DevAllocZ(&va, (size_t)rows * f->v_stride) &&
                  DevAllocZ(&vb, (size_t)rows * f->v_stride);
  f->d_va = reinterpret_cast<float*>(va);
  f->d_vb = reinterpret_cast<float*>(vb);
  if (!ok)
  {
    rfm_fir_destroy(f);
    return PFail(RFM_ERR_CUDA, "rfm_fir_create: device allocation failed");
  }
  *out = f;
  return RFM_OK;
}

void rfm_fir_destroy(rfm_fir* f)
{
  if (!f)
    return;
  cudaSetDevice(f->device);
  cudaFree(f->d_coef); cudaFree(f->d_va); cudaFree(f->d_vb); cudaFree(f->d_a); cudaFree(f->d_b); cudaFree(f->d_tmp);
  delete f;
}

// cFirFilter::InitLPFilter, FirFilter.cpp:78-148; *ntaps = its return value
int rfm_fir_init_lp(rfm_fir* f, uint32_t NumTaps, float Scale, float Astop, float Fpass, float Fstop, float Fs,
                    uint32_t* ntaps)
{
  if (!f)
    return PFail(RFM_ERR_INVALID, "rfm_fir_init_lp: null handle");
  cudaSetDevice(f->device);
  const std::vector<float> taps = PlanKaiserLP(NumTaps, Scale, Astop, Fpass, Fstop, Fs);
  if (ntaps)
    *ntaps = (uint32_t)taps.size();
  return FirInstall(f, taps);
}

// cFirFilter::InitHPFilter, FirFilter.cpp:195-264
int rfm_fir_init_hp(rfm_fir* f, uint32_t NumTaps, float Scale, float Astop, float Fpass, float Fstop, float Fs,
                    uint32_t* ntaps)
{
  if (!f)
    return PFail(RFM_ERR_INVALID, "rfm_fir_init_hp: null handle");
  cudaSetDevice(f->device);
  const std::vector<float> taps = PlanKaiserHP(NumTaps, Scale, Astop, Fpass, Fstop, Fs);
  if (ntaps)
    *ntaps = (uint32_t)taps.size();
  return FirInstall(f, taps);
}

// the two Kaiser designs on their own (host only, no device): kind 0 = InitLPFilter, 1 = InitHPFilter
int rfm_fir_design(int kind, uint32_t NumTaps, float Scale, float Astop, float Fpass, float Fstop, float Fs, float* out,
                   uint32_t max, uint32_t* n)
{
  if (!n || kind < 0 || kind > 1 || NumTaps > kMaxFirTaps)
    return PFail(RFM_ERR_INVALID, "rfm_fir_design: invalid argument");
  const std::vector<float> taps = kind == 0 ? PlanKaiserLP(NumTaps, Scale, Astop, Fpass, Fstop, Fs)
                                            : PlanKaiserHP(NumTaps, Scale, Astop, Fpass, Fstop, Fs);
  *n = (uint32_t)taps.size();
  for (size_t i = 0; out && i < taps.size() && i < max; ++i)
    out[i] = taps[i];
  return RFM_OK;
}

// cFirFilter::InitConstFir(NumTaps, const RealType*, Fsamprate), FirFilter.cpp:302-320
int rfm_fir_init_const(rfm_fir* f, uint32_t ntaps, const float* coef, float Fs)
{
  (void)Fs;
  if (!f || !coef)
    return PFail(RFM_ERR_INVALID, "rfm_fir_init_const: invalid argument");
  cudaSetDevice(f->device);
  return FirInstall(f, std::vector<float>(coef, coef + ntaps));
}

int rfm_fir_taps(const rfm_fir* f, float* out, uint32_t max, uint32_t* n)
{
  if (!f || !n)
    return PFail(RFM_ERR_INVALID, "rfm_fir_taps: invalid argument");
  *n = f->taps;
  for (unsigned i = 0; out && i < f->taps && i < max; ++i)
    out[i] = f->coef[i];
  return RFM_OK;
}

// mode 0: Process(RealType*), 1: Process(ComplexType*), 2: ProcessTwo(RealType*, RealType*); in place
int rfm_fir_process_device(rfm_fir* f, int mode, float* d_a, float* d_b, size_t stride, uint32_t n, void* cuda_stream)
{
  if (!f || !d_a || mode < 0 || mode > 2 || (mode == 2 && !d_b))
    return PFail(RFM_ERR_INVALID, "rfm_fir_process_device: invalid argument");
  if (f->taps == 0)
    return PFail(RFM_ERR_INVALID, "rfm_fir: filter not initialised");
  if (n > f->cap)
    return PFail(RFM_ERR_INVALID, "rfm_fir: n exceeds max_len");
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  const unsigned hist = f->taps - 1;
  const size_t vs_b = f->v_stride * sizeof(float2); // row pitch of the V buffers in bytes (either element size)
  dim3 grid((n + 255) / 256, f->rows);
  RotFirParams p;
  memset(&p, 0, sizeof(p));
  p.n = n; p.S = f->rows; p.taps = f->taps; p.g0 = f->g; p.coef = f->d_coef; p.out_off = 0;
  float* v = mode == 0 ? f->d_va : f->d_vb;
  const unsigned elem = mode == 0 ? 4 : 8;
  if (mode == 2)
  {
    if (!f->d_tmp && !DevAllocZ(&f->d_tmp, (size_t)f->rows * f->cap))
      return PFail(RFM_ERR_CUDA, "rfm_fir: scratch allocation failed");
    k_join_v<<<grid, 256, 0, st>>>(d_a, d_b, stride, reinterpret_cast<float2*>(v), f->v_stride, hist, n);
    p.outA = reinterpret_cast<float*>(f->d_tmp); p.out_stride = f->cap;
  }
  else
  {
    k_to_v<<<grid, 256, 0, st>>>(reinterpret_cast<const char*>(d_a), stride * elem, reinterpret_cast<char*>(v), vs_b, hist,
                                 n, elem);
    p.outA = d_a; p.out_stride = stride;
  }
  p.inA = v; p.inB = nullptr; p.in_stride = vs_b / elem; p.outB = nullptr; p.cplx = mode != 0;
  launch_rotfir(p, st);
  if (mode == 2)
    k_split<<<grid, 256, 0, st>>>(f->d_tmp, f->cap, d_a, d_b, stride, n);
  if (hist)
  {
    TailParams tp;
    tp.count = 0;
    tp.d[tp.count++] = {v, v, vs_b, hist, n, elem, f->rows};
    launch_tails(tp, f->rows, st);
  }
  f->g = (f->g + n) % f->taps;
  rfm::g_launches += 3;
  return cudaGetLastError() == cudaSuccess ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_fir: kernel launch failed");
}

static int FirHost(rfm_fir* f, int mode, float* a, float* b, uint32_t n)
{
  if (!f || !a || (mode == 2 && !b) || n > f->cap)
    return PFail(RFM_ERR_INVALID, "rfm_fir_process: invalid argument");
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  const size_t elems = (size_t)f->rows * f->cap * 2;
  if (!f->d_a && !DevAllocZ(&f->d_a, elems))
    return PFail(RFM_ERR_CUDA, "rfm_fir: staging allocation failed");
  if (mode == 2 && !f->d_b && !DevAllocZ(&f->d_b, elems))
    return PFail(RFM_ERR_CUDA, "rfm_fir: staging allocation failed");
  const size_t bytes = (size_t)f->rows * n * (mode == 1 ? 8 : 4);
  if (cudaMemcpy(f->d_a, a, bytes, cudaMemcpyHostToDevice) != cudaSuccess ||
      (mode == 2 && cudaMemcpy(f->d_b, b, bytes, cudaMemcpyHostToDevice) != cudaSuccess))
    return PFail(RFM_ERR_CUDA, "rfm_fir: H2D copy failed");
  int rc = rfm_fir_process_device(f, mode, f->d_a, f->d_b, n, n, nullptr);
  if (rc != RFM_OK)
    return rc;
  if (cudaMemcpy(a, f->d_a, bytes, cudaMemcpyDeviceToHost) != cudaSuccess ||
      (mode == 2 && cudaMemcpy(b, f->d_b, bytes, cudaMemcpyDeviceToHost) != cudaSuccess))
    return PFail(RFM_ERR_CUDA, "rfm_fir: D2H copy failed");
  return RFM_OK;
}

int rfm_fir_process_real(rfm_fir* f, float* buf, uint32_t n) { return FirHost(f, 0, buf, nullptr, n); }
int rfm_fir_process_complex(rfm_fir* f, float* buf, uint32_t n) { return FirHost(f, 1, buf, nullptr, n); }
int rfm_fir_process_two(rfm_fir* f, float* a, float* b, uint32_t n) { return FirHost(f, 2, a, b, n); }

} // extern "C"

// ==================================================================================================
// cRDSRxSignalProcessor
// ==================================================================================================
struct rfm_rdsproc
{
  unsigned rows = 0, cap = 0, nst = 0, nr_max = 0;
  int device = 0;
  DecoderPlan plan;
  unsigned hist[kRfMaxStages] = {0}, tail_off[kRfMaxStages + 1] = {0};
  unsigned tail_stride = 0, nr_stride = 0, mf_stride = 0, bits_cap = 0, min_n = 0;
  unsigned rlp_g = 0, mf_g = 0, pending = 0;
  float* d_taps[kRfMaxStages] = {nullptr};
  float *d_rlp = nullptr, *d_mf = nullptr, *d_osc1 = nullptr, *d_state = nullptr, *d_mfV = nullptr, *d_mf_out = nullptr;
  cf32 *d_osc = nullptr, *d_tails = nullptr, *d_rlp_out = nullptr;
  uint8_t* d_bits = nullptr;
  unsigned* d_count = nullptr;
  float* d_in = nullptr; // staging for the host entry point
  cudaStream_t last = nullptr;
  std::vector<RdsBlockSync> sync;
  std::vector<std::vector<uint8_t>> bits;
  std::vector<unsigned> h_counts;
  std::vector<uint8_t> h_bits;
};

namespace
{
constexpr size_t kMaxKeptBitsProc = 1u << 16;   // raw bits / groups retained per row between the take calls
constexpr size_t kMaxKeptGroupsProc = 4096;

int RdsDrain(rfm_rdsproc* r)
{
  if (r->pending == 0)
    return RFM_OK;
  if (cudaStreamSynchronize(r->last) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_rdsproc: stream synchronisation failed");
  r->h_counts.resize(r->rows);
  if (cudaMemcpy(r->h_counts.data(), r->d_count, r->rows * sizeof(unsigned), cudaMemcpyDeviceToHost) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_rdsproc: bit count read failed");
  unsigned mx = 0;
  for (unsigned c : r->h_counts)
    mx = std::max(mx, c);
  if (mx > r->bits_cap)
    return PFail(RFM_ERR_OVERFLOW, "rfm_rdsproc: bit buffer overflow");
  if (mx)
  {
    r->h_bits.resize((size_t)r->rows * mx);
    if (cudaMemcpy2D(r->h_bits.data(), mx, r->d_bits, r->bits_cap, mx, r->rows, cudaMemcpyDeviceToHost) != cudaSuccess)
      return PFail(RFM_ERR_CUDA, "rfm_rdsproc: bit read failed");
    for (unsigned s = 0; s < r->rows; ++s)
    {
      const uint8_t* b = r->h_bits.data() + (size_t)s * mx;
      r->bits[s].insert(r->bits[s].end(), b, b + r->h_counts[s]);
      if (r->bits[s].size() > kMaxKeptBitsProc) // bounded: a caller without a bit sink never takes them
        r->bits[s].erase(r->bits[s].begin(), r->bits[s].begin() + (r->bits[s].size() - kMaxKeptBitsProc));
      for (unsigned i = 0; i < r->h_counts[s]; ++i)
        r->sync[s].PushBit(b[i]); // ProcessNewRdsBit, RDSProcess.cpp:272-375
      auto& kept = r->sync[s].Groups();
      if (kept.size() > 4 * kMaxKeptGroupsProc)
        kept.erase(kept.begin(), kept.begin() + (kept.size() - 4 * kMaxKeptGroupsProc));
    }
    if (cudaMemset(r->d_count, 0, r->rows * sizeof(unsigned)) != cudaSuccess)
      return PFail(RFM_ERR_CUDA, "rfm_rdsproc: bit count reset failed");
  }
  r->pending = 0;
  return RFM_OK;
}

// cRDSRxSignalProcessor::Reset, RDSProcess.cpp:90-118 (the down-converter's oscillator and delay lines are NOT touched)
int RdsResetState(rfm_rdsproc* r)
{
  const unsigned S = r->rows;
  std::vector<float> st((size_t)SF_COUNT * S, 0.0f);
  bool ok = cudaMemcpy(r->d_state, st.data(), st.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
  const unsigned lp_hist = (unsigned)r->plan.rlp_coef.size() - 1;
  ok = ok && cudaMemset2D(r->d_tails + r->tail_off[r->nst], (size_t)r->tail_stride * sizeof(cf32), 0,
                          (size_t)lp_hist * sizeof(cf32), S) == cudaSuccess;
  ok = ok && cudaMemset(r->d_mfV, 0, (size_t)S * r->mf_stride * sizeof(float)) == cudaSuccess;
  r->rlp_g = 0;
  r->mf_g = 0;
  for (auto& s : r->sync)
    s.Reset();
  return ok ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_rdsproc: state reset failed");
}
} // namespace

extern "C"
{

int rfm_rdsproc_create(uint32_t rows, float sample_rate, uint32_t max_len, int device, rfm_rdsproc** out)
{
  if (!out || rows == 0 || max_len == 0 || !(sample_rate > 0))
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc_create: invalid argument");
  *out = nullptr;
  int rc = PickDevice(&device);
  if (rc != RFM_OK)
    return rc;
  rfm_rdsproc* r = new rfm_rdsproc;
  r->rows = rows; r->cap = max_len; r->device = device;
  // the constructor depends on the sample rate only (RDSProcess.cpp:43-88): the decoder planner with downsample = 1
  r->plan = PlanDecoder(sample_rate, 0.0, 48000.0, 15000.0, 1, false);
  const DecoderPlan& p = r->plan;
  r->nst = (unsigned)p.rds_stages.size();
  if (r->nst == 0 || r->nst > kRfMaxStages || p.mf_coef.size() < 2 || p.rlp_coef.size() > kMaxFirTapsDev)
  {
    delete r;
    return PFail(RFM_ERR_UNSUPPORTED, "rfm_rdsproc_create: sample rate outside the supported range");
  }
  unsigned off = 0;
  for (unsigned k = 0; k < r->nst; ++k)
  {
    const HalfBandStage& hs = p.rds_stages[k];
    r->hist[k] = hs.len == 3 ? 2u : (unsigned)hs.len - 1;
    r->tail_off[k] = off;
    off += r->hist[k];
    const unsigned need = hs.len == 3 ? 4u : (hs.fixed11 ? 20u : 2u * ((unsigned)hs.len - 1));
    r->min_n = std::max(r->min_n, need << k);
  }
  r->tail_off[r->nst] = off;
  off += (unsigned)p.rlp_coef.size() - 1;
  r->tail_stride = (off + 15u) & ~15u;
  r->nr_max = (max_len >> r->nst) + 1;
  r->nr_stride = (r->nr_max + 15u) & ~15u;
  r->mf_stride = ((unsigned)p.mf_coef.size() - 1 + r->nr_max + 15u) & ~15u;
  r->bits_cap = std::max(4096u, 2 * r->nr_max);
  bool ok = DevAllocZ(&r->d_rlp, p.rlp_coef.size()) && DevAllocZ(&r->d_mf, p.mf_coef.size()) && DevAllocZ(&r->d_osc1, 2) &&
            DevAllocZ(&r->d_state, (size_t)SF_COUNT * rows) && DevAllocZ(&r->d_mfV, (size_t)rows * r->mf_stride) &&
            DevAllocZ(&r->d_mf_out, (size_t)rows * r->nr_stride) && DevAllocZ(&r->d_osc, (size_t)max_len) &&
            DevAllocZ(&r->d_tails, (size_t)rows * r->tail_stride) && DevAllocZ(&r->d_rlp_out, (size_t)rows * r->nr_stride) &&
            DevAllocZ(&r->d_bits, (size_t)rows * r->bits_cap) && DevAllocZ(&r->d_count, rows);
  for (unsigned k = 0; ok && k < r->nst; ++k)
    if (p.rds_stages[k].h)
      ok = DevAllocZ(&r->d_taps[k], (size_t)p.rds_stages[k].len) &&
           cudaMemcpy(r->d_taps[k], p.rds_stages[k].h, p.rds_stages[k].len * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess;
  const float one[2] = {1.0f, 0.0f}; // DownConvert.cpp:283-284
  ok = ok && cudaMemcpy(r->d_rlp, p.rlp_coef.data(), p.rlp_coef.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess &&
       cudaMemcpy(r->d_mf, p.mf_coef.data(), p.mf_coef.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess &&
       cudaMemcpy(r->d_osc1, one, sizeof(one), cudaMemcpyHostToDevice) == cudaSuccess;
  r->sync.resize(rows);
  r->bits.resize(rows);
  if (!ok || RdsResetState(r) != RFM_OK)
  {
    rfm_rdsproc_destroy(r);
    return PFail(RFM_ERR_CUDA, "rfm_rdsproc_create: device allocation failed");
  }
  *out = r;
  return RFM_OK;
}

void rfm_rdsproc_destroy(rfm_rdsproc* r)
{
  if (!r)
    return;
  cudaSetDevice(r->device);
  for (auto* t : r->d_taps)
    cudaFree(t);
  cudaFree(r->d_rlp); cudaFree(r->d_mf); cudaFree(r->d_osc1); cudaFree(r->d_state); cudaFree(r->d_mfV);
  cudaFree(r->d_mf_out); cudaFree(r->d_osc); cudaFree(r->d_tails); cudaFree(r->d_rlp_out); cudaFree(r->d_bits);
  cudaFree(r->d_count); cudaFree(r->d_in);
  delete r;
}

float rfm_rdsproc_process_rate(const rfm_rdsproc* r) { return r ? r->plan.rds_rate : 0.0f; }

int rfm_rdsproc_reset(rfm_rdsproc* r)
{
  if (!r)
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc_reset: null handle");
  cudaSetDevice(r->device);
  int rc = RdsDrain(r); // bits sliced before the reset belong to the old state
  if (rc != RFM_OK)
    return rc;
  if (cudaDeviceSynchronize() != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_rdsproc_reset: synchronisation failed");
  return RdsResetState(r);
}

// cRDSRxSignalProcessor::Process(const RealType*, unsigned), RDSProcess.cpp:120-180; d_bb [rows][stride] on the device
int rfm_rdsproc_process_device(rfm_rdsproc* r, const float* d_bb, size_t stride, uint32_t n, void* cuda_stream)
{
  if (!r || !d_bb)
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc_process_device: invalid argument");
  if (n == 0)
    return RFM_OK;
  if (n > r->cap)
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc: n exceeds max_len");
  if (n % (1u << r->nst) != 0 || n < r->min_n)
    return PFail(RFM_ERR_UNSUPPORTED,
                 "rfm_rdsproc: n must be a multiple of 2^stages and give every half-band stage >= 2*(taps-1) samples "
                 "(the reference mis-filters such calls, DownConvert.cpp:519-520,544-547)");
  cudaSetDevice(r->device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  const DecoderPlan& p = r->plan;
  const unsigned S = r->rows, nr = n >> r->nst;
  const unsigned rlp_taps = (unsigned)p.rlp_coef.size(), mf_taps = (unsigned)p.mf_coef.size();
  if (r->pending + nr > r->bits_cap)
  {
    int rc = RdsDrain(r);
    if (rc != RFM_OK)
      return rc;
  }
  OscParams op;
  op.oscV = r->d_osc; op.osc_hist = 0; op.nb = n; op.osc1 = r->d_osc1; op.cosv = p.rds_osc.cosv; op.sinv = p.rds_osc.sinv;
  launch_osc(op, st);

  RdsFrontParams rf;
  memset(&rf, 0, sizeof(rf));
  rf.bbV = d_bb; rf.a_stride = stride; rf.a_hist = 0;
  rf.osc = r->d_osc; rf.nb = n; rf.S = S; rf.nst = r->nst;
  for (unsigned k = 0; k < r->nst; ++k)
  {
    const HalfBandStage& hs = p.rds_stages[k];
    rf.st[k].kind = hs.len == 3 ? 2 : (hs.fixed11 ? 1 : 0);
    rf.st[k].len = (unsigned)hs.len;
    rf.st[k].hist = r->hist[k];
    rf.st[k].h = r->d_taps[k];
    rf.tail_off[k] = r->tail_off[k];
  }
  rf.tail_off[r->nst] = r->tail_off[r->nst];
  rf.lp_coef = r->d_rlp; rf.lp_n = rlp_taps; rf.g0 = r->rlp_g;
  rf.tails = r->d_tails; rf.tail_stride = r->tail_stride;
  rf.out = r->d_rlp_out; rf.dec_out = nullptr; rf.out_stride = r->nr_stride;
  launch_rds_front(rf, st);

  RdsPllParams pp;
  pp.in = r->d_rlp_out; pp.in_stride = r->nr_stride; pp.nr = nr; pp.S = S; pp.state = r->d_state;
  pp.lo = p.rpll_lo; pp.hi = p.rpll_hi; pp.alpha = p.rpll_alpha; pp.beta = p.rpll_beta;
  pp.out = r->d_mfV; pp.out_stride = r->mf_stride; pp.out_off = mf_taps - 1;
  launch_rds_pll(pp, st);

  RotFirParams fmf;
  memset(&fmf, 0, sizeof(fmf));
  fmf.inA = r->d_mfV; fmf.inB = nullptr; fmf.in_stride = r->mf_stride; fmf.outA = r->d_mf_out; fmf.outB = nullptr;
  fmf.out_stride = r->nr_stride; fmf.out_off = 0; fmf.n = nr; fmf.S = S; fmf.taps = mf_taps; fmf.g0 = r->mf_g;
  fmf.coef = r->d_mf; fmf.cplx = 0;
  launch_rotfir(fmf, st);

  RdsSliceParams sp;
  sp.in = r->d_mf_out; sp.in_stride = r->nr_stride; sp.nr = nr; sp.S = S; sp.state = r->d_state;
  sp.sync = {p.rsync.A1, p.rsync.A2, p.rsync.B0, p.rsync.B1, p.rsync.B2};
  sp.bits = r->d_bits; sp.bits_cap = r->bits_cap; sp.bit_count = r->d_count;
  launch_rds_slice(sp, st);

  TailParams tp;
  tp.count = 0;
  tp.d[tp.count++] = {r->d_mfV, r->d_mfV, r->mf_stride * sizeof(float), mf_taps - 1, nr, 4, S};
  launch_tails(tp, S, st);

  r->rlp_g = (r->rlp_g + nr) % rlp_taps;
  r->mf_g = (r->mf_g + nr) % mf_taps;
  r->pending += nr;
  r->last = st;
  rfm::g_launches += 6;
  return cudaGetLastError() == cudaSuccess ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_rdsproc: kernel launch failed");
}

int rfm_rdsproc_process(rfm_rdsproc* r, const float* baseband, uint32_t n)
{
  if (!r || !baseband || n > r->cap)
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc_process: invalid argument");
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(r->device);
  if (!r->d_in && !DevAllocZ(&r->d_in, (size_t)r->rows * r->cap))
    return PFail(RFM_ERR_CUDA, "rfm_rdsproc: staging allocation failed");
  if (cudaMemcpy(r->d_in, baseband, (size_t)r->rows * n * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_rdsproc: H2D copy failed");
  int rc = rfm_rdsproc_process_device(r, r->d_in, n, n, nullptr);
  return rc == RFM_OK ? RdsDrain(r) : rc; // the host class delivers its bits inside Process, like the reference
}

int rfm_rdsproc_take_bits(rfm_rdsproc* r, uint32_t row, uint8_t* bits, uint32_t max_bits, uint32_t* n_bits)
{
  if (!r || row >= r->rows || !n_bits || (!bits && max_bits))
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc_take_bits: invalid argument");
  cudaSetDevice(r->device);
  int rc = RdsDrain(r);
  if (rc != RFM_OK)
    return rc;
  auto& b = r->bits[row];
  const uint32_t k = (uint32_t)std::min<size_t>(b.size(), max_bits);
  std::copy(b.begin(), b.begin() + k, bits);
  b.erase(b.begin(), b.begin() + k);
  *n_bits = k;
  return RFM_OK;
}

int rfm_rdsproc_take_groups(rfm_rdsproc* r, uint32_t row, uint16_t* groups, uint32_t max_groups, uint32_t* n_groups)
{
  if (!r || row >= r->rows || !n_groups || (!groups && max_groups))
    return PFail(RFM_ERR_INVALID, "rfm_rdsproc_take_groups: invalid argument");
  cudaSetDevice(r->device);
  int rc = RdsDrain(r);
  if (rc != RFM_OK)
    return rc;
  auto& g = r->sync[row].Groups();
  const uint32_t k = (uint32_t)std::min<size_t>(g.size() / 4, max_groups);
  std::copy(g.begin(), g.begin() + 4 * (size_t)k, groups);
  g.erase(g.begin(), g.begin() + 4 * (size_t)k);
  *n_groups = k;
  return RFM_OK;
}

} // extern "C"

// ==================================================================================================
// cDownsampleFilter (DownConvert.h:21-60, DownConvert.cpp:58-256): Lanczos-windowed sinc FIR with decimation.
// The two forms the chain uses: complex input with an integer factor (k_front, :98-154) and real input with a
// fractional factor (k_resample, :195-233).  Real + integer (:164-192, no caller in the reference) is a plain
// thread-per-output kernel below; complex + fractional is an endless loop in the reference (pstep == 0) and returns
// RFM_ERR_UNSUPPORTED.
// ==================================================================================================

// Real input, integer factor: y[i] = sum_{j = 1 .. order} x[p - j] c[j], p = pos + i ds, ascending j, every product and
// sum rounded on its own (DownConvert.cpp:172-190; both of its loops are this sum over V = [history(order) | block],
// x[p - j] = V[order + p - j]).  Thread per output, taps in shared memory; not on the hot path, so no window staging.
namespace
{
__global__ void __launch_bounds__(128) k_downsample_real_int(const float* __restrict__ v, size_t v_stride,
                                                             const float* __restrict__ coeff, unsigned order, unsigned ds,
                                                             unsigned pos, unsigned nout, float* __restrict__ out,
                                                             size_t out_stride)
{
  extern __shared__ float s_c[]; // c[0 .. order]
  for (unsigned j = threadIdx.x; j <= order; j += 128)
    s_c[j] = coeff[j];
  __syncthreads();
  const unsigned i = blockIdx.x * 128 + threadIdx.x;
  if (i >= nout)
    return;
  const float* x = v + (size_t)blockIdx.y * v_stride + order + pos + (size_t)i * ds;
  float y = 0.0f;
  for (unsigned j = 1; j <= order; ++j)
    y = addf(y, mulf(x[-(int)j], s_c[j]));
  out[(size_t)blockIdx.y * out_stride + i] = y;
}
} // namespace

struct rfm_downsample
{
  unsigned rows = 0, cap = 0, order = 0, ds_int = 0;
  int device = 0;
  bool integer = true;
  double downsample = 1.0;
  float pstep = 1.0f, pos_frac = 0.0f;
  unsigned pos_int = 0;
  std::vector<float> coeff;
  float *d_coeff = nullptr, *d_lut = nullptr, *d_v = nullptr, *d_scratch = nullptr;
  cf32* d_tail = nullptr;
  size_t v_stride = 0;
  float *d_in = nullptr, *d_out = nullptr; // staging for the host entry points
};

extern "C"
{

int rfm_downsample_create(uint32_t rows, uint32_t filter_order, double cutoff, double downsample, int integer_factor,
                          uint32_t max_len, int device, rfm_downsample** out)
{
  if (!out || rows == 0 || max_len == 0 || filter_order < 2 || filter_order > 512 || !(downsample >= 1.0))
    return PFail(RFM_ERR_INVALID, "rfm_downsample_create: invalid argument");
  *out = nullptr;
  int rc = PickDevice(&device);
  if (rc != RFM_OK)
    return rc;
  rfm_downsample* f = new rfm_downsample;
  f->rows = rows; f->cap = max_len; f->order = filter_order; f->device = device;
  f->integer = integer_factor != 0;
  f->downsample = downsample;
  f->ds_int = f->integer ? (unsigned)lrint(downsample) : 0; // DownConvert.cpp:68
  f->pstep = (float)downsample;                             // :203 RealType pstep = m_downsample
  f->coeff = PlanLanczos(filter_order, cutoff);             // :78 (order + 2 entries)
  f->v_stride = ((size_t)filter_order + max_len + 15) & ~(size_t)15;
  std::vector<float> lut(256);
  for (int u = 0; u < 256; ++u)
    lut[u] = (float)(u / (255.0 / 2.0) - 1.0);
  bool ok = DevAllocZ(&f->d_coeff, f->coeff.size()) && DevAllocZ(&f->d_lut, 256) &&
            DevAllocZ(&f->d_tail, (size_t)rows * filter_order) && DevAllocZ(&f->d_v, (size_t)rows * f->v_stride) &&
            DevAllocZ(&f->d_scratch, (size_t)rows * (max_len + 16));
  ok = ok && cudaMemcpy(f->d_coeff, f->coeff.data(), f->coeff.size() * sizeof(float), cudaMemcpyHostToDevice) == cudaSuccess &&
       cudaMemcpy(f->d_lut, lut.data(), 1024, cudaMemcpyHostToDevice) == cudaSuccess;
  if (!ok)
  {
    rfm_downsample_destroy(f);
    return PFail(RFM_ERR_CUDA, "rfm_downsample_create: device allocation failed");
  }
  *out = f;
  return RFM_OK;
}

void rfm_downsample_destroy(rfm_downsample* f)
{
  if (!f)
    return;
  cudaSetDevice(f->device);
  cudaFree(f->d_coeff); cudaFree(f->d_lut); cudaFree(f->d_tail); cudaFree(f->d_v); cudaFree(f->d_scratch);
  cudaFree(f->d_in); cudaFree(f->d_out);
  delete f;
}

int rfm_downsample_reset(rfm_downsample* f) // DownConvert.cpp:90-96
{
  if (!f)
    return PFail(RFM_ERR_INVALID, "rfm_downsample_reset: null handle");
  cudaSetDevice(f->device);
  f->pos_int = 0;
  f->pos_frac = 0.0f;
  const bool ok = cudaMemsetAsync(f->d_tail, 0, (size_t)f->rows * f->order * sizeof(cf32), 0) == cudaSuccess &&
                  cudaMemsetAsync(f->d_v, 0, (size_t)f->rows * f->v_stride * sizeof(float), 0) == cudaSuccess;
  return ok ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_downsample_reset: failed");
}

int rfm_downsample_coefficients(const rfm_downsample* f, float* out, uint32_t max, uint32_t* n)
{
  if (!f || !n)
    return PFail(RFM_ERR_INVALID, "rfm_downsample_coefficients: invalid argument");
  *n = (uint32_t)f->coeff.size();
  for (size_t i = 0; out && i < f->coeff.size() && i < max; ++i)
    out[i] = f->coeff[i];
  return RFM_OK;
}

uint32_t rfm_downsample_max_outputs(const rfm_downsample* f, uint32_t n)
{
  if (!f)
    return 0;
  return (uint32_t)((double)n / (f->integer ? (double)f->ds_int : f->downsample)) + 2;
}

// unsigned Process(const ComplexType* in, ComplexType* out, unsigned length), DownConvert.cpp:98-154
int rfm_downsample_process_complex_device(rfm_downsample* f, const float* d_in, size_t in_stride, float* d_out,
                                          size_t out_stride, uint32_t n, uint32_t* n_out, void* cuda_stream)
{
  if (n_out)
    *n_out = 0;
  if (!f || !d_in || !d_out)
    return PFail(RFM_ERR_INVALID, "rfm_downsample_process_complex_device: invalid argument");
  if (!f->integer || f->ds_int == 0)
    return PFail(RFM_ERR_UNSUPPORTED, "cDownsampleFilter: the complex overload needs an integer factor "
                                      "(the reference loops forever otherwise, DownConvert.cpp:108-112)");
  if (n == 0)
    return RFM_OK;
  if (n > f->cap)
    return PFail(RFM_ERR_INVALID, "rfm_downsample: n exceeds max_len");
  if (n < f->order)
    return PFail(RFM_ERR_UNSUPPORTED, "rfm_downsample: calls shorter than the filter order are not supported");
  cudaSetDevice(f->device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  const unsigned pos = f->pos_int, ds = f->ds_int;
  const unsigned nout = pos < n ? (n - pos + ds - 1) / ds : 0;
  FrontParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.in = d_in; fp.in_stride = in_stride; fp.n = n; fp.S = f->rows; fp.order = f->order; fp.ds = ds;
  fp.p0 = pos; fp.nout = nout; fp.idx0 = 0; fp.lut = f->d_lut; fp.tuner = nullptr;
  fp.coeff = f->d_coeff; fp.coeff_host = nullptr; // generic kernel (the tiled one has the fine tuner built in)
  fp.tail = f->d_tail; fp.z = reinterpret_cast<cf32*>(d_out); fp.z_stride = out_stride;
  launch_front(fp, kIqCF32, st);
  launch_front_tail(fp, kIqCF32, st);
  f->pos_int = pos + nout * ds - n; // :132
  rfm::g_launches += 2;
  if (n_out)
    *n_out = nout;
  return cudaGetLastError() == cudaSuccess ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_downsample: kernel launch failed");
}

// unsigned Process(const RealType* in, RealType* out, unsigned length), fractional branch, DownConvert.cpp:195-256
int rfm_downsample_process_real_device(rfm_downsample* f, const float* d_in, size_t in_stride, float* d_out,
                                       size_t out_stride, uint32_t n, uint32_t* n_out, void* cuda_stream)
{
  if (n_out)
    *n_out = 0;
  if (!f || !d_in || !d_out)
    return PFail(RFM_ERR_INVALID, "rfm_downsample_process_real_device: invalid argument");
  if (n == 0)
    return RFM_OK;
  if (n > f->cap)
    return PFail(RFM_ERR_INVALID, "rfm_downsample: n exceeds max_len");
  if (n < f->order)
    return PFail(RFM_ERR_UNSUPPORTED, "rfm_downsample: calls shorter than the filter order are not supported");
  cudaSetDevice(f->device);
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  if (f->integer) // DownConvert.cpp:164-192
  {
    if (f->ds_int == 0)
      return PFail(RFM_ERR_INVALID, "rfm_downsample: integer factor of 0");
    const unsigned pos = f->pos_int, ds = f->ds_int;
    const unsigned nout = pos < n ? (n - pos + ds - 1) / ds : 0;
    if (nout > out_stride)
      return PFail(RFM_ERR_INVALID, "rfm_downsample: out_stride is shorter than the output");
    dim3 grid((n + 255) / 256, f->rows);
    k_to_v<<<grid, 256, 0, st>>>(reinterpret_cast<const char*>(d_in), in_stride * 4, reinterpret_cast<char*>(f->d_v),
                                 f->v_stride * 4, f->order, n, 4);
    if (nout)
      k_downsample_real_int<<<dim3((nout + 127) / 128, f->rows), 128, (f->order + 1) * sizeof(float), st>>>(
          f->d_v, f->v_stride, f->d_coeff, f->order, ds, pos, nout, d_out, out_stride);
    TailParams tp;
    tp.count = 0;
    tp.d[tp.count++] = {f->d_v, f->d_v, f->v_stride * 4, f->order, n, 4, f->rows};
    launch_tails(tp, f->rows, st);
    f->pos_int = pos + nout * ds - n; // :192
    rfm::g_launches += 3;
    if (n_out)
      *n_out = nout;
    return cudaGetLastError() == cudaSuccess ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_downsample: kernel launch failed");
  }
  float pos_next = 0.0f;
  const unsigned na = FractionalOutputs(f->pos_frac, f->pstep, n, &pos_next);
  dim3 grid((n + 255) / 256, f->rows);
  k_to_v<<<grid, 256, 0, st>>>(reinterpret_cast<const char*>(d_in), in_stride * 4, reinterpret_cast<char*>(f->d_v),
                               f->v_stride * 4, f->order, n, 4);
  ResampleParams rp;
  memset(&rp, 0, sizeof(rp));
  rp.bbV = f->d_v; rp.rawV = f->d_v; rp.a_stride = f->v_stride; rp.order = f->order; rp.nb = n; rp.S = f->rows;
  rp.na = na; rp.pos_frac = f->pos_frac; rp.pstep = f->pstep; rp.coeff = f->d_coeff;
  rp.lpM = d_out; rp.lpS = f->d_scratch; rp.lp_stride = out_stride; rp.lp_hist = 0;
  if (out_stride > (size_t)f->cap + 16)
    return PFail(RFM_ERR_INVALID, "rfm_downsample: out_stride exceeds max_len + 16");
  launch_resample(rp, st);
  TailParams tp;
  tp.count = 0;
  tp.d[tp.count++] = {f->d_v, f->d_v, f->v_stride * 4, f->order, n, 4, f->rows};
  launch_tails(tp, f->rows, st);
  f->pos_frac = pos_next;
  rfm::g_launches += 3;
  if (n_out)
    *n_out = na;
  return cudaGetLastError() == cudaSuccess ? RFM_OK : PFail(RFM_ERR_CUDA, "rfm_downsample: kernel launch failed");
}

static int DownsampleHost(rfm_downsample* f, bool cplx, const float* in, float* out, uint32_t n, uint32_t* n_out)
{
  if (!f || !in || !out || n > f->cap)
    return PFail(RFM_ERR_INVALID, "rfm_downsample_process: invalid argument");
  if (n_out)
    *n_out = 0;
  if (n == 0)
    return RFM_OK;
  cudaSetDevice(f->device);
  const size_t cap_out = (size_t)f->cap + 16;
  if (!f->d_in && !DevAllocZ(&f->d_in, (size_t)f->rows * f->cap * 2))
    return PFail(RFM_ERR_CUDA, "rfm_downsample: staging allocation failed");
  if (!f->d_out && !DevAllocZ(&f->d_out, (size_t)f->rows * cap_out * 2))
    return PFail(RFM_ERR_CUDA, "rfm_downsample: staging allocation failed");
  const size_t esz = cplx ? 8 : 4;
  if (cudaMemcpy(f->d_in, in, (size_t)f->rows * n * esz, cudaMemcpyHostToDevice) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_downsample: H2D copy failed");
  uint32_t m = 0;
  int rc = cplx ? rfm_downsample_process_complex_device(f, f->d_in, n, f->d_out, cap_out, n, &m, nullptr)
                : rfm_downsample_process_real_device(f, f->d_in, n, f->d_out, cap_out, n, &m, nullptr);
  if (rc != RFM_OK)
    return rc;
  // rows are compacted on the way back: out is [rows][m]
  if (m && cudaMemcpy2D(out, (size_t)m * esz, f->d_out, cap_out * esz, (size_t)m * esz, f->rows, cudaMemcpyDeviceToHost) != cudaSuccess)
    return PFail(RFM_ERR_CUDA, "rfm_downsample: D2H copy failed");
  if (n_out)
    *n_out = m;
  return RFM_OK;
}

int rfm_downsample_process_complex(rfm_downsample* f, const float* in, float* out, uint32_t n, uint32_t* n_out)
{
  return DownsampleHost(f, true, in, out, n, n_out);
}
int rfm_downsample_process_real(rfm_downsample* f, const float* in, float* out, uint32_t n, uint32_t* n_out)
{
  return DownsampleHost(f, false, in, out, n, n_out);
}

} // extern "C"
