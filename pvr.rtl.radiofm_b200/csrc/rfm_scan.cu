// rfm_scan.cu -- band scan of one wideband capture (u8, s8, s16 or cf32): which FM stations does it hold, how strong are they, and what
// do they identify as.  The reference's tuner dialog answers this one frequency at a time (ChannelSettings.cpp:96-147:
// retune, wait, cFmDecoder::StereoDetected); here every channel of the capture is decided in one pass.
//
//   1. averaged power spectrum (k_scan_psd + k_scan_reduce): Welch, N = 4096 periodic-Hann segments, hop N/2, radix-4
//      Stockham FFT in shared memory; each CTA owns kScanSegsPerCta consecutive segments and writes one partial row,
//      the rows are summed in row order in double -- no atomics, so the result is independent of the device, its SM
//      count and any SM partition.
//   2. channels (host, double): the raster's bins, channel powers, the 25th-percentile noise floor, local maxima at
//      least min_snr_db above it.
//   3. confirmation: the reference's receiver on every candidate, composed exactly as wideband.py composes it with the
//      "osc" mixer -- rfm_downconvert (CRDSDownConvert::SetFrequency(-f) + SetWfmDataRate, shared capture) feeding one
//      rfm_decoder (cFmDecoder(rate, 0, 48000, 15000, 1)) per call of 16000 baseband samples, the front end of call
//      k+1 overlapping the demodulator of call k; then status, RDS groups, PI and the name cRDSGroupDecoder publishes.
//      rfm_scan_set_mixer(RFM_SCAN_MIXER_NCO) composes the "nco" receiver instead: rows at 0 Hz behind the phasor NCO.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <string>
#include <vector>

#include "../../include/radiofm_b200.h"
#include "rfm_dsp.cuh"
#include "rfm_kernels.cuh"
#include "rfm_plan.h"

namespace rfm
{
extern std::atomic<uint64_t> g_launches;
void SetLastError(const std::string& m);
int IqEstimateDevice(int fmt, const void* d_in, uint64_t n, cudaStream_t st, rfm_iq_correction* out);  // rfm_iqcorr.cu
int IqEstimateCheck(const char* who, int fmt, const void* iq, uint64_t n, bool on_device);
}

namespace
{
constexpr unsigned kScanN = 4096;          // segment length, fixed (not an option)
constexpr unsigned kScanHop = kScanN / 2;
constexpr unsigned kScanThreads = 256;
constexpr unsigned kScanPerThread = kScanN / kScanThreads;
constexpr unsigned kScanSegsPerCta = 32;   // set by n alone: the partial rows do not depend on the device
constexpr unsigned kScanSmem = 2 * kScanN * sizeof(float2);   // Stockham ping-pong, 64 KB
constexpr uint32_t kScanCallBb = 16000;    // baseband samples per demodulator call (wideband.py: 64 x 32000 >> 7)
constexpr float kScanMaxBw = 100000.0f;    // CRDSDownConvert::SetWfmDataRate bandwidth, as in wideband.py
constexpr unsigned kScanSlots = 3;         // wideband.py n_slots

int ScanFail(int code, const std::string& m)
{
  rfm::SetLastError(m);
  return code;
}

// One radix-4 Stockham pass (decimation in frequency, self-sorting): sub-transform length n = N / 4^ST, stride
// s = 4^ST.  Butterfly t = q + s p reads x[t + m N/4] (m = 0..3) and writes y[q + s (4p + m)]; the twiddles
// w^(m p s) = exp(-2 pi j m p s / N) come from the host-made table tw[k] = (cos, sin)(2 pi k / N).
template <int ST>
__device__ __forceinline__ void ScanPass(const float2* __restrict__ x, float2* __restrict__ y,
                                         const float2* __restrict__ tw, unsigned tid)
{
  constexpr unsigned s = 1u << (2 * ST);
  constexpr unsigned q4 = kScanN / 4;
#pragma unroll
  for (unsigned b = 0; b < kScanN / 4 / kScanThreads; ++b)
  {
    const unsigned t = tid + b * kScanThreads;
    const unsigned q = t & (s - 1);
    const unsigned ps = t - q;                       // p * s
    const float2 a = x[t], bb = x[t + q4], c = x[t + 2 * q4], d = x[t + 3 * q4];
    const float2 apc = make_float2(a.x + c.x, a.y + c.y), amc = make_float2(a.x - c.x, a.y - c.y);
    const float2 bpd = make_float2(bb.x + d.x, bb.y + d.y), bmd = make_float2(bb.x - d.x, bb.y - d.y);
    // j (b - d) = (-bmd.y, bmd.x)
    const float2 u1 = make_float2(amc.x + bmd.y, amc.y - bmd.x);
    const float2 u2 = make_float2(apc.x - bpd.x, apc.y - bpd.y);
    const float2 u3 = make_float2(amc.x - bmd.y, amc.y + bmd.x);
    const unsigned o = q + 4 * ps;
    y[o] = make_float2(apc.x + bpd.x, apc.y + bpd.y);
    if (ST == 5)
    {
      y[o + s] = u1;
      y[o + 2 * s] = u2;
      y[o + 3 * s] = u3;
    }
    else
    {
      const float2 w1 = __ldg(tw + ps), w2 = __ldg(tw + 2 * ps), w3 = __ldg(tw + 3 * ps);
      // u * conj(w)
      y[o + s] = make_float2(u1.x * w1.x + u1.y * w1.y, u1.y * w1.x - u1.x * w1.y);
      y[o + 2 * s] = make_float2(u2.x * w2.x + u2.y * w2.y, u2.y * w2.x - u2.x * w2.y);
      y[o + 3 * s] = make_float2(u3.x * w3.x + u3.y * w3.y, u3.y * w3.x - u3.x * w3.y);
    }
  }
}

// One capture sample of IqFormat F (rfm_dsp.cuh): its storage type and its value as float
template <int F> struct ScanIn { using T = unsigned short; };   // u8, s8: one byte each for I and Q
template <> struct ScanIn<rfm::kIqS16> { using T = unsigned; };
template <> struct ScanIn<rfm::kIqCF32> { using T = float2; };
__device__ __forceinline__ float2 ScanSample(unsigned w)
{
  return make_float2(rfm::rfm_s16_to_float(w, 0u), rfm::rfm_s16_to_float(w, 1u));
}
__device__ __forceinline__ float2 ScanSample(float2 v)
{
  return v;
}

// Partial Welch sums: CTA b transforms segments [b * 32, b * 32 + 32) of the capture (I,Q samples of format F; segment g
// covers samples [g N/2, g N/2 + N)) and writes sum |X_g[k]|^2 over them, natural bin order, to partial[b][k].
// CORR: every sample is IQ-corrected (rfm_iq_correct) after its conversion, before the window.
template <int F, bool CORR>
__global__ void __launch_bounds__(kScanThreads) k_scan_psd(const typename ScanIn<F>::T* __restrict__ cap, uint64_t n_seg,
                                                           const float* __restrict__ win, const float2* __restrict__ tw,
                                                           float* __restrict__ partial, rfm::IqCorr corr)
{
  extern __shared__ float2 scan_sm[];
  float2* A = scan_sm;
  float2* B = scan_sm + kScanN;
  const unsigned tid = threadIdx.x;
  const uint64_t g0 = (uint64_t)blockIdx.x * kScanSegsPerCta;
  const uint64_t g1 = min(g0 + kScanSegsPerCta, n_seg);
  float acc[kScanPerThread];
#pragma unroll
  for (unsigned j = 0; j < kScanPerThread; ++j)
    acc[j] = 0.0f;
  for (uint64_t g = g0; g < g1; ++g)
  {
    const typename ScanIn<F>::T* seg = cap + g * kScanHop;
    if constexpr (F == rfm::kIqU8 || F == rfm::kIqS8)
    {
#pragma unroll
      for (unsigned j = 0; j < kScanPerThread; ++j)
      {
        const unsigned i = tid + j * kScanThreads;
        const unsigned w = __ldg(seg + i);
        const float h = __ldg(win + i);
        if constexpr (CORR)
        {
          const float2 x = rfm::rfm_iq_correct(
              make_float2(rfm::rfm_iq8_to_float<F>(w, 0u), rfm::rfm_iq8_to_float<F>(w, 1u)), corr);
          A[i] = make_float2(h * x.x, h * x.y);
        }
        else
          A[i] = make_float2(h * rfm::rfm_iq8_to_float<F>(w, 0u), h * rfm::rfm_iq8_to_float<F>(w, 1u));
      }
    }
    else
    {
      // partly unrolled: fully unrolled, the wider loads of the whole segment were hoisted into 190 registers
#pragma unroll 4
      for (unsigned j = 0; j < kScanPerThread; ++j)
      {
        const unsigned i = tid + j * kScanThreads;
        float2 x = ScanSample(__ldg(seg + i));
        if (CORR)
          x = rfm::rfm_iq_correct(x, corr);
        const float h = __ldg(win + i);
        A[i] = make_float2(h * x.x, h * x.y);
      }
    }
    __syncthreads();
    ScanPass<0>(A, B, tw, tid);
    __syncthreads();
    ScanPass<1>(B, A, tw, tid);
    __syncthreads();
    ScanPass<2>(A, B, tw, tid);
    __syncthreads();
    ScanPass<3>(B, A, tw, tid);
    __syncthreads();
    ScanPass<4>(A, B, tw, tid);
    __syncthreads();
    ScanPass<5>(B, A, tw, tid);
    __syncthreads();
#pragma unroll
    for (unsigned j = 0; j < kScanPerThread; ++j)
    {
      const float2 v = A[tid + j * kScanThreads];
      acc[j] += v.x * v.x + v.y * v.y;
    }
    __syncthreads();
  }
  float* row = partial + (size_t)blockIdx.x * kScanN;
#pragma unroll
  for (unsigned j = 0; j < kScanPerThread; ++j)
    row[tid + j * kScanThreads] = acc[j];
}

// P[k] = (sum over the partial rows, in row order, in double) / (S N sum w^2), written centred (index N/2 = 0 Hz).
__global__ void __launch_bounds__(kScanThreads) k_scan_reduce(const float* __restrict__ partial, unsigned rows,
                                                              double norm, float* __restrict__ psd)
{
  const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= kScanN)
    return;
  double acc = 0.0;
  for (unsigned r = 0; r < rows; ++r)
    acc += (double)partial[(size_t)r * kScanN + k];
  psd[(k + kScanN / 2) & (kScanN - 1)] = (float)(acc / norm);
}

template <typename T>
cudaError_t DevAlloc(T** p, size_t n)
{
  return cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T));
}

// Bin centre frequency of centred index k, Hz from the capture centre.  oracle/scan.py evaluates the same expressions.
double BinFreq(unsigned k, double fs) { return (double)((int)k - (int)(kScanN / 2)) * fs / (double)kScanN; }
double RasterFreq(const rfm_scan_config& c, unsigned j) { return c.raster_first + (double)j * c.raster_step; }
} // namespace

struct rfm_scan
{
  rfm_scan_config cfg;
  int device = 0;
  unsigned stages = 0;
  uint32_t n_call = 0;
  std::vector<uint32_t> bin_lo, bin_hi;   // channel j owns centred bins [bin_lo[j], bin_hi[j])
  cudaStream_t st = nullptr;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  float* d_win = nullptr;
  float2* d_tw = nullptr;
  uint8_t* d_cap = nullptr;               // staging for host input
  size_t cap_bytes = 0;
  float* d_partial = nullptr;
  size_t partial_rows = 0;
  float* d_psd = nullptr;
  double sum_w2 = 0.0;
  bool have = false;
  std::vector<float> psd;
  std::vector<double> chan;
  std::vector<rfm_scan_station> stations;
  double spectrum_ms = 0.0, confirm_ms = 0.0;
  int corr_mode = 0;                      // rfm_scan_set_iq_correction
  rfm_iq_correction corr_fixed = {0.f, 0.f, 1.f, 0.f, 0};
  rfm_iq_correction corr_applied = {0.f, 0.f, 1.f, 0.f, 0};
  int mixer = RFM_SCAN_MIXER_OSC;         // rfm_scan_set_mixer
};

namespace
{
// The candidates' receivers: one rfm_downconvert row and one rfm_decoder stream per candidate, `calls` calls of
// n_call capture samples each, the front end on the decoder's companion stream, three baseband slots.
int Confirm(rfm_scan* s, int fmt, const uint8_t* d_cap, uint64_t calls, const std::vector<uint32_t>& cand,
            const rfm_iq_correction* corr)
{
  const uint32_t M = (uint32_t)cand.size();
  const bool pnco = s->mixer == RFM_SCAN_MIXER_NCO;
  std::vector<float> nco(M, 0.0f);
  std::vector<double> pnco_freq(M);
  for (uint32_t m = 0; m < M; ++m)
  {
    pnco_freq[m] = -RasterFreq(s->cfg, cand[m]);
    if (!pnco)
      nco[m] = (float)pnco_freq[m];
  }
  rfm_downconvert* dc = nullptr;
  rfm_decoder* dec = nullptr;
  cudaStream_t s_dec = nullptr, s_done = nullptr;
  cudaEvent_t ev_bb = nullptr, ev_free[kScanSlots] = {};
  float2* bb[kScanSlots] = {};
  float* audio[kScanSlots] = {};
  int rc = rfm_downconvert_create(M, nco.data(), (float)s->cfg.sample_rate, kScanMaxBw, 1, s->n_call, s->device, &dc);
  if (rc == RFM_OK)
    rc = rfm_downconvert_set_iq_correction(dc, corr);
  if (rc == RFM_OK && pnco)
    rc = rfm_downconvert_set_nco(dc, pnco_freq.data());
  size_t stride = 0;
  void* front = nullptr;
  if (rc == RFM_OK)
  {
    rfm_config c;
    rfm_config_default(&c);
    c.sample_rate_if = rfm_downconvert_output_rate(dc);
    c.tuning_offset = 0.0;
    c.sample_rate_pcm = 48000.0;
    c.bandwidth_pcm = 15000.0;
    c.downsample = 1;
    c.n_streams = M;
    c.max_block_len = kScanCallBb;
    c.device = s->device;
    c.lanes_sms = 8;
    rc = rfm_decoder_create(&c, &dec);
  }
  if (rc == RFM_OK)
    rc = rfm_decoder_companion_stream(dec, &front);
  if (rc == RFM_OK)
  {
    stride = std::max<size_t>(rfm_decoder_max_audio_floats(dec, kScanCallBb), 2);
    stride = (stride + 1) & ~(size_t)1;
    bool ok = cudaStreamCreateWithFlags(&s_dec, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&s_done, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&ev_bb, cudaEventDisableTiming) == cudaSuccess;
    for (unsigned k = 0; ok && k < kScanSlots; ++k)
      ok = cudaEventCreateWithFlags(&ev_free[k], cudaEventDisableTiming) == cudaSuccess &&
           DevAlloc(&bb[k], (size_t)M * kScanCallBb) == cudaSuccess &&
           DevAlloc(&audio[k], (size_t)M * stride) == cudaSuccess;
    if (!ok)
      rc = ScanFail(RFM_ERR_CUDA, "rfm_scan: confirmation set-up failed");
  }
  if (rc == RFM_OK)
  {
    cudaEventRecord(s->ev[2], s_dec);
    cudaStreamWaitEvent((cudaStream_t)front, s->ev[2], 0);
    for (uint64_t k = 0; rc == RFM_OK && k < calls; ++k)
    {
      const unsigned slot = (unsigned)(k % kScanSlots);
      if (k >= kScanSlots)
        cudaStreamWaitEvent((cudaStream_t)front, ev_free[slot], 0);   // the slot's previous call has left the decoder
      uint32_t m = 0, na = 0;
      rc = rfm_downconvert_process_iq_device(dc, fmt, 1, d_cap + rfm::IqBytes(fmt) * k * (uint64_t)s->n_call, s->n_call,
                                             reinterpret_cast<float*>(bb[slot]), kScanCallBb, s->n_call, &m, front);
      if (rc == RFM_OK && m != kScanCallBb)
        rc = ScanFail(RFM_ERR_CUDA, "rfm_scan: unexpected front-end output length");
      if (rc != RFM_OK)
        break;
      cudaEventRecord(ev_bb, (cudaStream_t)front);
      cudaStreamWaitEvent(s_dec, ev_bb, 0);
      rc = rfm_decoder_process_cf32_device(dec, reinterpret_cast<const float*>(bb[slot]), kScanCallBb, kScanCallBb,
                                           audio[slot], stride, &na, s_dec);
      if (rc == RFM_OK)
        rc = rfm_decoder_wait(dec, s_done);
      cudaEventRecord(ev_free[slot], s_done);
    }
    cudaEventRecord(s->ev[3], s_done);
    if (rc == RFM_OK)
      rc = rfm_decoder_synchronize(dec);
    if (rc == RFM_OK && cudaStreamSynchronize(s_done) != cudaSuccess)
      rc = ScanFail(RFM_ERR_CUDA, "rfm_scan: confirmation failed");
    float ms = 0.0f;
    if (rc == RFM_OK && cudaEventElapsedTime(&ms, s->ev[2], s->ev[3]) == cudaSuccess)
      s->confirm_ms = ms;
  }
  std::vector<uint16_t> groups, buf(4 * 4096);
  for (uint32_t m = 0; rc == RFM_OK && m < M; ++m)
  {
    rfm_scan_station& o = s->stations[m];
    rfm_stream_status stt;
    rc = rfm_decoder_get_status(dec, m, &stt);
    if (rc != RFM_OK)
      break;
    o.stereo_detected = stt.stereo_detected;
    o.pilot_level = stt.pilot_level;
    o.interface_level = stt.interface_level;
    o.baseband_level = stt.baseband_level;
    groups.clear();
    uint32_t ng = 0;
    do
    {
      rc = rfm_decoder_rds_take_groups(dec, m, buf.data(), 4096, &ng);
      groups.insert(groups.end(), buf.begin(), buf.begin() + 4 * (size_t)ng);
    } while (rc == RFM_OK && ng == 4096);
    if (rc != RFM_OK)
      break;
    const uint32_t n_groups = (uint32_t)(groups.size() / 4);
    o.rds_groups = n_groups;
    // PI: the most frequent block A, ties to the value seen first
    std::map<uint16_t, std::pair<uint32_t, uint32_t>> count;   // value -> (count, first position)
    for (uint32_t g = 0; g < n_groups; ++g)
    {
      auto it = count.find(groups[4 * g]);
      if (it == count.end())
        count[groups[4 * g]] = {1u, g};
      else
        ++it->second.first;
    }
    o.pi = -1;
    uint32_t best = 0, best_pos = 0;
    for (const auto& kv : count)
      if (kv.second.first > best || (kv.second.first == best && kv.second.second < best_pos))
      {
        best = kv.second.first;
        best_pos = kv.second.second;
        o.pi = kv.first;
      }
    // PS: the reference's naming path, cRDSGroupDecoder -> cRadioReceiver::SetChannelName
    rfm_rdsgroup* rg = nullptr;
    rc = rfm_rdsgroup_create(nullptr, &rg);
    if (rc == RFM_OK)
      rc = rfm_rdsgroup_decode(rg, groups.data(), n_groups);
    if (rc == RFM_OK)
      rc = rfm_rdsgroup_channel_name(rg, o.ps);
    o.ps[8] = 0;
    rfm_rdsgroup_destroy(rg);
  }
  for (unsigned k = 0; k < kScanSlots; ++k)
  {
    cudaFree(bb[k]);
    cudaFree(audio[k]);
    if (ev_free[k])
      cudaEventDestroy(ev_free[k]);
  }
  if (ev_bb)
    cudaEventDestroy(ev_bb);
  if (s_dec)
    cudaStreamDestroy(s_dec);
  if (s_done)
    cudaStreamDestroy(s_done);
  rfm_decoder_destroy(dec);
  rfm_downconvert_destroy(dc);
  return rc;
}
} // namespace

extern "C"
{

void rfm_scan_config_default(rfm_scan_config* cfg)
{
  if (!cfg)
    return;
  memset(cfg, 0, sizeof(*cfg));
  cfg->sample_rate = 2.4e6;          // the add-on's RTL-SDR rate
  cfg->raster_first = -1.1e6;
  cfg->raster_step = 100000.0;
  cfg->raster_count = 23;
  cfg->min_snr_db = 10.0;
  cfg->device = -1;
}

int rfm_scan_create(const rfm_scan_config* cfg, rfm_scan** out)
{
  if (!cfg || !out)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_create: null argument");
  *out = nullptr;
  const double fs = cfg->sample_rate;
  if (!(fs > 0.0) || !isfinite(fs) || !isfinite(cfg->raster_first) || !isfinite(cfg->raster_step) ||
      !isfinite(cfg->min_snr_db))
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_create: sample rate, raster and min_snr_db must be finite");
  if (!(cfg->raster_step >= 4.0 * fs / kScanN))
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_create: raster_step below 4 spectrum bins (4 Fs / 4096)");
  if (cfg->raster_count < 1 || cfg->raster_count > kScanN)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_create: raster_count must be 1 .. 4096");
  for (unsigned j = 0; j < cfg->raster_count; ++j)
    if (fabs(RasterFreq(*cfg, j)) + 100000.0 > fs / 2.0)
      return ScanFail(RFM_ERR_INVALID, "rfm_scan_create: a raster channel reaches beyond the capture (|f| + 100 kHz > Fs/2)");
  std::vector<rfm::HalfBandStage> stages;
  rfm::PlanDecimationChain((float)fs, kScanMaxBw, true, &stages);
  if (stages.empty())
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_create: the WFM decimation chain has no stage at this rate (<= 400 kHz)");
  if (stages.size() > 9 || (uint64_t)kScanCallBb << stages.size() > 0xFFFFFFFFull)
    return ScanFail(RFM_ERR_UNSUPPORTED, "rfm_scan_create: more than 9 decimation stages (rfm_downconvert's limit)");

  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return ScanFail(RFM_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  int dev = cfg->device;
  if (dev < 0 && cudaGetDevice(&dev) != cudaSuccess)
    return ScanFail(RFM_ERR_CUDA, "cudaGetDevice failed");
  if (dev >= ndev)
    return ScanFail(RFM_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess)
    return ScanFail(RFM_ERR_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return ScanFail(RFM_ERR_NO_DEVICE, std::string("kernels are built for sm_100a only; device is ") + prop.name);
  if (cudaSetDevice(dev) != cudaSuccess)
    return ScanFail(RFM_ERR_CUDA, "cudaSetDevice failed");

  rfm_scan* s = new rfm_scan;
  s->cfg = *cfg;
  s->device = dev;
  s->stages = (unsigned)stages.size();
  s->n_call = kScanCallBb << s->stages;
  // raster point j owns the bins whose centre f satisfies f_j - step/2 <= f < f_j + step/2 (both bounds are monotone
  // in k, so each is a boundary found by stepping from an estimate)
  const double step = cfg->raster_step;
  auto first_at_or_above = [&](double f) {
    long k = (long)floor(f / fs * kScanN) + (long)(kScanN / 2);
    k = std::min<long>(std::max<long>(k, 0), kScanN);
    auto in = [&](long i) { return BinFreq((unsigned)i, fs) >= f; };
    while (k > 0 && in(k - 1))
      --k;
    while (k < (long)kScanN && !in(k))
      ++k;
    return (uint32_t)k;
  };
  for (unsigned j = 0; j < cfg->raster_count; ++j)
  {
    const double fj = RasterFreq(*cfg, j);
    s->bin_lo.push_back(first_at_or_above(fj - step / 2));
    s->bin_hi.push_back(std::max(s->bin_lo.back(), first_at_or_above(fj + step / 2)));
  }
  std::vector<float> win(kScanN), tw(2 * kScanN);
  for (unsigned i = 0; i < kScanN; ++i)
  {
    const double a = 2.0 * M_PI * (double)i / (double)kScanN;
    const double w = 0.5 - 0.5 * cos(a);
    win[i] = (float)w;
    s->sum_w2 += w * w;
    tw[2 * i] = (float)cos(a);
    tw[2 * i + 1] = (float)sin(a);
  }
  bool ok = cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking) == cudaSuccess;
  for (auto& e : s->ev)
    ok = ok && cudaEventCreate(&e) == cudaSuccess;
  ok = ok && DevAlloc(&s->d_win, kScanN) == cudaSuccess && DevAlloc(&s->d_tw, kScanN) == cudaSuccess &&
       DevAlloc(&s->d_psd, kScanN) == cudaSuccess &&
       cudaMemcpyAsync(s->d_win, win.data(), kScanN * sizeof(float), cudaMemcpyHostToDevice, s->st) == cudaSuccess &&
       cudaMemcpyAsync(s->d_tw, tw.data(), kScanN * sizeof(float2), cudaMemcpyHostToDevice, s->st) == cudaSuccess &&
       cudaStreamSynchronize(s->st) == cudaSuccess;
  if (!ok)
  {
    rfm_scan_destroy(s);
    return ScanFail(RFM_ERR_CUDA, "rfm_scan_create: device set-up failed");
  }
  *out = s;
  return RFM_OK;
}

void rfm_scan_destroy(rfm_scan* s)
{
  if (!s)
    return;
  cudaSetDevice(s->device);
  if (s->st)
    cudaStreamSynchronize(s->st);
  cudaFree(s->d_win);
  cudaFree(s->d_tw);
  cudaFree(s->d_cap);
  cudaFree(s->d_partial);
  cudaFree(s->d_psd);
  for (auto e : s->ev)
    if (e)
      cudaEventDestroy(e);
  if (s->st)
    cudaStreamDestroy(s->st);
  delete s;
}

int rfm_scan_run_u8(rfm_scan* s, const uint8_t* iq, uint64_t n, int iq_on_device)
{
  return rfm_scan_run(s, RFM_IQ_U8, iq, n, iq_on_device);
}

int rfm_scan_run(rfm_scan* s, int format, const void* iq, uint64_t n, int iq_on_device)
{
  if (!s || !iq)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_run: null argument");
  const uint32_t esz = rfm_iq_format_bytes(format);
  if (esz == 0)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_run: unknown IQ format");
  if (n < s->n_call)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_run: the capture is shorter than one demodulator call");
  if (iq_on_device && (reinterpret_cast<uintptr_t>(iq) % esz) != 0)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_run: device capture must be aligned to the sample size "
                                     "(2 / 2 / 4 / 8 bytes for u8 / s8 / s16 / cf32)");
  if (s->corr_mode == 1)
  {
    const int rc = rfm::IqEstimateCheck("rfm_scan_run", format, iq, n, iq_on_device != 0);
    if (rc != RFM_OK)
      return rc;
  }
  if (cudaSetDevice(s->device) != cudaSuccess)
    return ScanFail(RFM_ERR_CUDA, "cudaSetDevice failed");
  s->have = false;
  const uint8_t* d_cap = static_cast<const uint8_t*>(iq);
  if (!iq_on_device)
  {
    if (s->cap_bytes < esz * n)
    {
      cudaFree(s->d_cap);
      s->d_cap = nullptr;
      s->cap_bytes = 0;
      if (DevAlloc(&s->d_cap, esz * n) != cudaSuccess)
        return ScanFail(RFM_ERR_CUDA, "rfm_scan_run: capture allocation failed");
      s->cap_bytes = esz * n;
    }
    if (cudaMemcpyAsync(s->d_cap, iq, esz * n, cudaMemcpyHostToDevice, s->st) != cudaSuccess)
      return ScanFail(RFM_ERR_CUDA, "rfm_scan_run: H2D copy failed");
    d_cap = s->d_cap;
  }
  // 1. spectrum
  const uint64_t n_seg = (n - kScanN) / kScanHop + 1;
  const uint64_t rows = (n_seg + kScanSegsPerCta - 1) / kScanSegsPerCta;
  if (rows > 0x7FFFFFFFull)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_run: capture too long");
  if (s->partial_rows < rows)
  {
    cudaFree(s->d_partial);
    s->d_partial = nullptr;
    s->partial_rows = 0;
    if (DevAlloc(&s->d_partial, (size_t)rows * kScanN) != cudaSuccess)
      return ScanFail(RFM_ERR_CUDA, "rfm_scan_run: partial-spectrum allocation failed");
    s->partial_rows = rows;
  }
  cudaEventRecord(s->ev[0], s->st);
  // IQ correction: the statistics pass (mode 1) runs inside the spectrum's timed stage
  s->corr_applied = rfm_iq_correction{0.f, 0.f, 1.f, 0.f, 0};
  if (s->corr_mode == 1)
  {
    const int rc = rfm::IqEstimateDevice(format, d_cap, n, s->st, &s->corr_applied);
    if (rc != RFM_OK)
      return rc;
  }
  else if (s->corr_mode == 2)
    s->corr_applied = s->corr_fixed;
  const bool corr_on = s->corr_mode != 0;
  const rfm::IqCorr corr = {s->corr_applied.dc_i, s->corr_applied.dc_q, s->corr_applied.a, s->corr_applied.b};
#define RFM_SCAN_PSD_C(F, C)                                                                                            \
  rfm::EnsureDynSmem(k_scan_psd<F, C>, kScanSmem);                                                                      \
  k_scan_psd<F, C><<<(unsigned)rows, kScanThreads, kScanSmem, s->st>>>(                                                 \
      reinterpret_cast<const typename ScanIn<F>::T*>(d_cap), n_seg, s->d_win, s->d_tw, s->d_partial, corr)
#define RFM_SCAN_PSD(F)                                                                                                 \
  if (corr_on)                                                                                                          \
  {                                                                                                                     \
    RFM_SCAN_PSD_C(F, true);                                                                                            \
  }                                                                                                                     \
  else                                                                                                                  \
  {                                                                                                                     \
    RFM_SCAN_PSD_C(F, false);                                                                                           \
  }
  switch (format)
  {
    case RFM_IQ_U8: RFM_SCAN_PSD(rfm::kIqU8); break;
    case RFM_IQ_S8: RFM_SCAN_PSD(rfm::kIqS8); break;
    case RFM_IQ_S16: RFM_SCAN_PSD(rfm::kIqS16); break;
    default: RFM_SCAN_PSD(rfm::kIqCF32); break;
  }
#undef RFM_SCAN_PSD
#undef RFM_SCAN_PSD_C
  k_scan_reduce<<<kScanN / kScanThreads, kScanThreads, 0, s->st>>>(s->d_partial, (unsigned)rows,
                                                                   (double)n_seg * (double)kScanN * s->sum_w2, s->d_psd);
  cudaEventRecord(s->ev[1], s->st);
  rfm::g_launches += 2;
  if (cudaGetLastError() != cudaSuccess)
    return ScanFail(RFM_ERR_CUDA, "rfm_scan: spectrum kernel launch failed");
  s->psd.assign(kScanN, 0.0f);
  if (cudaMemcpyAsync(s->psd.data(), s->d_psd, kScanN * sizeof(float), cudaMemcpyDeviceToHost, s->st) != cudaSuccess ||
      cudaStreamSynchronize(s->st) != cudaSuccess)
    return ScanFail(RFM_ERR_CUDA, std::string("rfm_scan: spectrum failed: ") + cudaGetErrorString(cudaGetLastError()));
  float ms = 0.0f;
  cudaEventElapsedTime(&ms, s->ev[0], s->ev[1]);
  s->spectrum_ms = ms;
  s->confirm_ms = 0.0;

  // 2. channels, floor, candidates
  const unsigned count = s->cfg.raster_count;
  s->chan.assign(count, 0.0);
  for (unsigned j = 0; j < count; ++j)
    for (uint32_t k = s->bin_lo[j]; k < s->bin_hi[j]; ++k)
      s->chan[j] += (double)s->psd[k];
  std::vector<double> sorted(s->chan);
  std::sort(sorted.begin(), sorted.end());
  const double floor_c = sorted[(count - 1) / 4];
  const double thr = floor_c * pow(10.0, s->cfg.min_snr_db / 10.0);
  std::vector<uint32_t> cand;
  for (unsigned j = 0; j < count; ++j)
  {
    const double c = s->chan[j];
    if (c >= thr && (j == 0 || c > s->chan[j - 1]) && (j + 1 == count || c >= s->chan[j + 1]))
      cand.push_back(j);
  }
  s->stations.assign(cand.size(), rfm_scan_station{});
  for (size_t m = 0; m < cand.size(); ++m)
  {
    rfm_scan_station& o = s->stations[m];
    o.freq = RasterFreq(s->cfg, cand[m]);
    o.power_dbfs = (float)(10.0 * log10(s->chan[cand[m]]));
    o.snr_db = (float)(10.0 * log10(s->chan[cand[m]] / floor_c));
    o.pi = -1;
  }

  // 3. confirmation over every whole call of the capture
  if (!cand.empty())
  {
    const int rc = Confirm(s, format, d_cap, n / s->n_call, cand, corr_on ? &s->corr_applied : nullptr);
    if (rc != RFM_OK)
    {
      s->stations.clear();
      return rc;
    }
  }
  s->have = true;
  return RFM_OK;
}

int rfm_scan_spectrum(rfm_scan* s, float* psd, uint32_t max, uint32_t* n_bins)
{
  if (!s || !n_bins || !s->have)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_spectrum: no completed run");
  *n_bins = kScanN;
  if (!psd || max < kScanN)
    return ScanFail(RFM_ERR_OVERFLOW, "rfm_scan_spectrum: buffer smaller than 4096 bins");
  memcpy(psd, s->psd.data(), kScanN * sizeof(float));
  return RFM_OK;
}

int rfm_scan_channel_power(rfm_scan* s, double* out, uint32_t max)
{
  if (!s || !out || !s->have)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_channel_power: no completed run");
  if (max < s->cfg.raster_count)
    return ScanFail(RFM_ERR_OVERFLOW, "rfm_scan_channel_power: buffer smaller than raster_count");
  memcpy(out, s->chan.data(), s->chan.size() * sizeof(double));
  return RFM_OK;
}

int rfm_scan_stations(rfm_scan* s, rfm_scan_station* out, uint32_t max, uint32_t* n)
{
  if (!s || !n || !s->have)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_stations: no completed run");
  *n = (uint32_t)s->stations.size();
  if (*n > max || (*n && !out))
    return ScanFail(RFM_ERR_OVERFLOW, "rfm_scan_stations: buffer too small");
  if (*n)
    memcpy(out, s->stations.data(), *n * sizeof(rfm_scan_station));
  return RFM_OK;
}

int rfm_scan_set_iq_correction(rfm_scan* s, int mode, const rfm_iq_correction* fixed)
{
  if (!s)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_set_iq_correction: null handle");
  if (mode < 0 || mode > 2)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_set_iq_correction: unknown mode (0 off, 1 estimate, 2 fixed)");
  if (mode == 2 && !fixed)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_set_iq_correction: mode 2 needs the fixed coefficients (NULL given)");
  if (mode == 2 && !(isfinite(fixed->dc_i) && isfinite(fixed->dc_q) && isfinite(fixed->a) && isfinite(fixed->b)))
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_set_iq_correction: coefficients must be finite");
  s->corr_mode = mode;
  if (mode == 2)
    s->corr_fixed = *fixed;
  return RFM_OK;
}

int rfm_scan_set_mixer(rfm_scan* s, int mixer)
{
  if (!s)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_set_mixer: null handle");
  if (mixer != RFM_SCAN_MIXER_OSC && mixer != RFM_SCAN_MIXER_NCO)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_set_mixer: unknown mixer (0 osc, 1 nco)");
  s->mixer = mixer;
  return RFM_OK;
}

int rfm_scan_iq_correction(rfm_scan* s, rfm_iq_correction* out)
{
  if (!s || !out || !s->have)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_iq_correction: no completed run");
  *out = s->corr_applied;
  return RFM_OK;
}

int rfm_scan_timing(rfm_scan* s, double* spectrum_ms, double* confirm_ms)
{
  if (!s || !s->have)
    return ScanFail(RFM_ERR_INVALID, "rfm_scan_timing: no completed run");
  if (spectrum_ms)
    *spectrum_ms = s->spectrum_ms;
  if (confirm_ms)
    *confirm_ms = s->confirm_ms;
  return RFM_OK;
}

} // extern "C"
