// rfm_api.cu -- C ABI (include/radiofm_b200.h) over the sm_100a kernels: decoder handle, HBM buffers,
// per-block launch schedule, stream-group pipelining, RDS bit drain.
//
// Execution model.  One decoder = n_streams independent IQ streams processed in lock step, split into G groups
// (G = 1 unless asked otherwise; the host-pointer entry points use groups to overlap H2D / compute / D2H).
// Each group owns three CUDA streams and runs every block as a three-stage software pipeline:
//     stage F (stream sF):  if_level, front (IQ format -> float -> tune -> FIR / ds), time-parallel FM-demodulator PLL
//     stage A (stream sA, high priority):  bb_lanes (DC tracker / meters || pilot PLL)
//     stage B (stream sB):  { resample -> lp29 -> audio_tail }, { halfband* -> rds lp -> rds pll -> matched
//                           filter -> slicer }, tails
// While the lanes of block k run, the front end of block k+1 and stage B of block k-1 are in flight: the
// one-lane-per-stream PLL kernel (nonlinear recurrences, latency-bound, 2 warps per SM) is the long pole and hides
// the throughput-bound FIR kernels.  Everything handed from one stage to the next (decimated IQ, baseband / L-R
// rows, stereo flag) is double-buffered by block parity; the NCO-oscillator table of the RDS mixer (identical for
// all streams) is produced ahead on its own stream.
#include <cuda.h> // declarations only: the green-context entry points are looked up at run time (libcuda is not linked)
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/radiofm_b200.h"
#include "rfm_dsp.cuh"
#include "rfm_kernels.cuh"
#include "rfm_plan.h"
#include "rfm_rdsgroup.h"
#include "rfm_rdssync.h"

using namespace rfm;

namespace rfm
{
// shared with the stand-alone primitives (rfm_downconvert.cu, rfm_filters.cu)
std::atomic<uint64_t> g_launches{0};
thread_local std::string g_err;
void SetLastError(const std::string& m) { g_err = m; }
} // namespace rfm

namespace
{
int Fail(int code, const std::string& msg)
{
  g_err = msg;
  return code;
}

#define RFM_CUDA(expr)                                                                                   \
  do                                                                                                     \
  {                                                                                                      \
    cudaError_t e_ = (expr);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return Fail(RFM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));                    \
  } while (0)

constexpr size_t kMaxKeptBits = 1u << 16; // raw RDS bits retained per stream between rfm_decoder_rds_take_bits calls
constexpr size_t kMaxKeptGroups = 4096;   // decoded groups retained per stream between rfm_decoder_rds_take_groups calls (6 min)

unsigned AlignUp(unsigned v, unsigned a) { return (v + a - 1) / a * a; }

template <typename T>
struct DevBuf
{
  T* p = nullptr;
  size_t n = 0;
  cudaError_t Alloc(size_t count)
  {
    n = count;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess)
      e = cudaMemset(p, 0, std::max<size_t>(count, 1) * sizeof(T));
    return e;
  }
  void Free()
  {
    if (p)
      cudaFree(p);
    p = nullptr;
  }
};

// Optional per-kernel timing: CUDA event pairs recorded around every launch on the stream the kernel is
// launched on (bench.py's roofline leg).  Off by default.
constexpr int kMaxProfKinds = 24;
struct ProfSlot
{
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;
  size_t used = 0;
};

struct Group
{
  unsigned s0 = 0, S = 0;
  ProfSlot prof[kMaxProfKinds];
  // front / lanes / resamplers / audio tail (LP, deemphasis, notch, matrix, D2H) / RDS front / RDS PLL + slicer
  cudaStream_t sF = nullptr, sA = nullptr, sB = nullptr, sC = nullptr, sR = nullptr, sP = nullptr;
  cudaStream_t* AllStreams(cudaStream_t (&v)[6]) const
  {
    v[0] = sF; v[1] = sA; v[2] = sB; v[3] = sC; v[4] = sR; v[5] = sP;
    return v;
  }
  cudaEvent_t ev_rds[3] = {nullptr, nullptr, nullptr};  // RDS front of the block finished (mod 3): bbV / oscV released
  cudaEvent_t ev_res[2] = {nullptr, nullptr};   // resamplers of the block with this parity finished: lpS / lpM [parity] written
  cudaEvent_t ev_aud[3] = {nullptr, nullptr, nullptr}; // audio tail ... finished (its stereo-flag slot, by block index mod 3, may be rewritten)
  cudaEvent_t ev_carry[2] = {nullptr, nullptr}; // LP history carried out of lpS / lpM [parity ^ 1]: they may be overwritten
  cudaEvent_t ev_pll[2] = {nullptr, nullptr};   // RDS PLL + slicer ... finished: rlp_out[parity] may be overwritten
  cudaEvent_t ev_front[2] = {nullptr, nullptr}; // front end of the block with this parity finished
  cudaEvent_t ev_demod[2] = {nullptr, nullptr}; // demodulator done: z[parity] may be overwritten
  cudaEvent_t ev_lanes[2] = {nullptr, nullptr}; // PLL lanes ...
  cudaEvent_t ev_rest[3] = {nullptr, nullptr, nullptr}; // stage B ... (by block index mod 3)
  DevBuf<cf32> tail, z[2];
  DevBuf<float> incr[2];       // NCO increments, demodulator (stage F) -> lanes (stage A), by parity
  DevBuf<float2> dm_start, dm_end; // speculative demodulator chunk states
  DevBuf<float> bbV[3], rawV[3]; // lanes -> stage B hand-over: three deep, so stage B of block k has two lane periods
  DevBuf<cf32> rlpV, rlp_out[2]; // rlpV: decimator output of the last block (stage tap); rlp_out: RDS LP output, by parity
  DevBuf<cf32> rds_tails;       // fused RDS front: per-stream histories of every stage + LP delay line
  DevBuf<float> mfV, mf_out;
  DevBuf<uint8_t> bits;
  DevBuf<unsigned> bit_count;
  DevBuf<float> lpS[2], lpM[2], fS, fM; // resampler outputs ([history | block], by parity); audio LP outputs
  DevBuf<float> state;
  DevBuf<uint8_t> in_stage;  // host-API staging of the input block
  DevBuf<float> audio_stage; // host-API staging of the audio block
};
} // namespace

// Experimental SM partition (RFM_LANES_SMS=N, N a multiple of 8): the stream of the latency-bound lanes kernel lives in
// a green context of N SMs, every other stream in a green context of the remaining SMs, so the pilot recurrence does
// not wait for issue slots behind the FIR kernels (DESIGN.md section 4).  Placement only: kernels and results unchanged.
struct SmPartition
{
  CUgreenCtx lanes = nullptr, rest = nullptr;
  unsigned lanes_sms = 0, rest_sms = 0;
};

struct rfm_decoder
{
  SmPartition part;
  rfm_config cfg;
  DecoderPlan plan;
  int device = 0;
  unsigned S = 0, maxn = 0;
  unsigned nb_max = 0, na_max = 0, nr_max = 0;
  unsigned z_stride = 0, a_stride = 0, lp_stride = 0, rlp_stride = 0, mf_stride = 0, nr_stride = 0;
  unsigned hb_stride[kMaxDecStages] = {0};
  unsigned osc_hist = 0, bits_cap = 0, audio_cap = 0;
  unsigned rds_tail_stride = 0, rds_tail_off[kRfMaxStages + 1] = {0};
  // plan tables on the device
  DevBuf<float> d_lut, d_tuner, d_in_coeff, d_a_coeff, d_lp_coef, d_rlp_coef, d_mf_coef;
  DevBuf<float> d_hb[kMaxDecStages];
  DevBuf<cf32> oscV[3];
  DevBuf<float> osc1;
  DevBuf<unsigned long long> d_repairs; // demodulator chunks repaired sequentially (telemetry)
  DevBuf<float> res_kk[3]; // per-block interpolated resampler taps, shared by all streams (by block index mod 3)
  DevBuf<int> res_meta[3];
  unsigned res_lp = 0;
  cudaStream_t s_osc = nullptr;
  cudaStream_t s_companion = nullptr; // rfm_decoder_companion_stream: created on first use
  cudaEvent_t ev_osc[3] = {nullptr, nullptr, nullptr};
  uint64_t block_index = 0; // blocks enqueued so far; parity selects the double buffers
  std::vector<Group> groups;
  bool profiling = false;
  const char* prof_names[kMaxProfKinds] = {nullptr};
  double prof_ms[kMaxProfKinds] = {0};
  uint64_t prof_count[kMaxProfKinds] = {0};
  ProfSlot main_prof[kMaxProfKinds];
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_base = nullptr;
  // lock-step state (identical for every stream)
  unsigned tuner_idx = 0, in_pos = 0;
  float a_pos = 0.0f;
  unsigned lp_g = 0, rlp_g = 0, mf_g = 0;
  unsigned pending_bits_bound = 0; // worst-case undrained bits per stream
  // geometry of the last block (for taps)
  unsigned last_n = 0, last_nb = 0, last_na = 0, last_nr = 0;
  unsigned last_nb_rds = 0; // baseband samples the RDS branch took from the last block (0 when it was skipped)
  unsigned last_hb_n[kMaxDecStages + 1] = {0};
  // host RDS state
  std::vector<RdsBlockSync> sync;
  std::vector<RdsGroupDecoder> uecp; // per stream: groups -> UECP byte stream; rfm_decoder_reset resets them (RDSProcess.cpp:92)
  std::vector<std::vector<uint8_t>> host_bits;
  uint8_t* h_drain = nullptr; // pinned staging of the drained bit counts + bits of every stream
  size_t h_drain_cap = 0;
};

namespace
{

template <typename F>
bool DriverEntry(const char* name, F* fn)
{
  void* f = nullptr;
  cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
  if (cudaGetDriverEntryPoint(name, &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !f)
  {
    cudaGetLastError();
    return false;
  }
  *fn = reinterpret_cast<F>(f);
  return true;
}

// false (with a reason) when the driver cannot do it: the caller then stays on ordinary streams
bool MakeSmPartition(int device, unsigned lanes_sms, SmPartition* out, std::string* why)
{
  decltype(&cuDeviceGet) p_get = nullptr;
  decltype(&cuDeviceGetDevResource) p_res = nullptr;
  decltype(&cuDevSmResourceSplitByCount) p_split = nullptr;
  decltype(&cuDevResourceGenerateDesc) p_desc = nullptr;
  decltype(&cuGreenCtxCreate) p_create = nullptr;
  if (!DriverEntry("cuDeviceGet", &p_get) || !DriverEntry("cuDeviceGetDevResource", &p_res) ||
      !DriverEntry("cuDevSmResourceSplitByCount", &p_split) || !DriverEntry("cuDevResourceGenerateDesc", &p_desc) ||
      !DriverEntry("cuGreenCtxCreate", &p_create))
  {
    *why = "green-context entry points not available in this driver";
    return false;
  }
  CUdevice dev;
  CUdevResource all, part, rest;
  unsigned groups = 1;
  CUdevResourceDesc d_part, d_rest;
  CUresult rc;
  if ((rc = p_get(&dev, device)) != CUDA_SUCCESS || (rc = p_res(dev, &all, CU_DEV_RESOURCE_TYPE_SM)) != CUDA_SUCCESS ||
      (rc = p_split(&part, &groups, &all, &rest, 0, lanes_sms)) != CUDA_SUCCESS || groups != 1 ||
      (rc = p_desc(&d_part, &part, 1)) != CUDA_SUCCESS || (rc = p_desc(&d_rest, &rest, 1)) != CUDA_SUCCESS ||
      (rc = p_create(&out->lanes, d_part, dev, CU_GREEN_CTX_DEFAULT_STREAM)) != CUDA_SUCCESS ||
      (rc = p_create(&out->rest, d_rest, dev, CU_GREEN_CTX_DEFAULT_STREAM)) != CUDA_SUCCESS)
  {
    *why = "SM partition failed, CUresult " + std::to_string((int)rc);
    return false;
  }
  out->lanes_sms = part.sm.smCount;
  out->rest_sms = rest.sm.smCount;
  return true;
}

// a stream of priority `prio`: in the given green context when the decoder is partitioned, an ordinary one otherwise
cudaError_t MakeStream(CUgreenCtx ctx, cudaStream_t* st, int prio)
{
  if (!ctx)
    return cudaStreamCreateWithPriority(st, cudaStreamNonBlocking, prio);
  decltype(&cuGreenCtxStreamCreate) p_stream = nullptr;
  if (!DriverEntry("cuGreenCtxStreamCreate", &p_stream))
    return cudaErrorNotSupported;
  CUstream cs = nullptr;
  if (p_stream(&cs, ctx, CU_STREAM_NON_BLOCKING, prio) != CUDA_SUCCESS)
    return cudaErrorUnknown;
  *st = cs;
  return cudaSuccess;
}

void FreeSmPartition(SmPartition* p)
{
  decltype(&cuGreenCtxDestroy) p_destroy = nullptr;
  if ((p->lanes || p->rest) && DriverEntry("cuGreenCtxDestroy", &p_destroy))
  {
    if (p->lanes)
      p_destroy(p->lanes);
    if (p->rest)
      p_destroy(p->rest);
  }
  p->lanes = p->rest = nullptr;
}

void ProfFree(ProfSlot* slots);

void FreeDecoder(rfm_decoder* d)
{
  if (!d)
    return;
  cudaSetDevice(d->device);
  for (auto& g : d->groups)
  {
    cudaStream_t all[6];
    g.AllStreams(all);
    for (cudaStream_t st : all)
      if (st)
        cudaStreamSynchronize(st);
    g.tail.Free(); g.z[0].Free(); g.z[1].Free(); g.incr[0].Free(); g.incr[1].Free(); g.dm_start.Free(); g.dm_end.Free();
    for (int b = 0; b < 3; ++b)
    {
      g.bbV[b].Free();
      g.rawV[b].Free();
    }
    g.rlpV.Free(); g.rlp_out[0].Free(); g.rlp_out[1].Free(); g.rds_tails.Free(); g.mfV.Free(); g.mf_out.Free(); g.bits.Free(); g.bit_count.Free();
    g.lpS[0].Free(); g.lpS[1].Free(); g.lpM[0].Free(); g.lpM[1].Free(); g.fS.Free(); g.fM.Free(); g.state.Free(); g.in_stage.Free(); g.audio_stage.Free();
    ProfFree(g.prof);
    for (cudaEvent_t e : {g.ev_demod[0], g.ev_demod[1], g.ev_front[0], g.ev_front[1], g.ev_lanes[0], g.ev_lanes[1], g.ev_rest[0], g.ev_rest[1], g.ev_rest[2], g.ev_rds[0], g.ev_rds[1], g.ev_rds[2],
                          g.ev_res[0], g.ev_res[1], g.ev_aud[0], g.ev_aud[1], g.ev_aud[2], g.ev_pll[0], g.ev_pll[1], g.ev_carry[0], g.ev_carry[1]})
      if (e)
        cudaEventDestroy(e);
    if (g.sF == g.sA)
      g.sF = g.sB = g.sC = g.sR = g.sP = nullptr; // RFM_DEBUG_SERIAL aliasing
    g.AllStreams(all);
    for (cudaStream_t st : all)
      if (st)
        cudaStreamDestroy(st);
  }
  d->d_lut.Free(); d->d_tuner.Free(); d->d_in_coeff.Free(); d->d_a_coeff.Free(); d->d_lp_coef.Free();
  d->d_rlp_coef.Free(); d->d_mf_coef.Free();
  for (auto& b : d->d_hb) b.Free();
  if (d->s_osc)
    cudaStreamSynchronize(d->s_osc);
  d->oscV[0].Free(); d->oscV[1].Free(); d->oscV[2].Free(); d->osc1.Free(); d->d_repairs.Free();
  for (int b = 0; b < 3; ++b)
  {
    d->res_kk[b].Free();
    d->res_meta[b].Free();
  }
  ProfFree(d->main_prof);
  for (cudaEvent_t e : {d->ev_fork, d->ev_osc[0], d->ev_osc[1], d->ev_osc[2], d->ev_join})
    if (e)
      cudaEventDestroy(e);
  if (d->s_osc)
    cudaStreamDestroy(d->s_osc);
  if (d->s_companion)
    cudaStreamDestroy(d->s_companion);
  if (d->h_drain)
    cudaFreeHost(d->h_drain);
  FreeSmPartition(&d->part);
  delete d;
}

cudaError_t Upload(DevBuf<float>& b, const float* src, size_t n)
{
  cudaError_t e = b.Alloc(n);
  if (e == cudaSuccess && n)
    e = cudaMemcpy(b.p, src, n * sizeof(float), cudaMemcpyHostToDevice);
  return e;
}

int ProfKind(rfm_decoder* d, const char* name)
{
  for (int i = 0; i < kMaxProfKinds; ++i)
  {
    if (!d->prof_names[i])
    {
      d->prof_names[i] = name;
      return i;
    }
    if (d->prof_names[i] == name || strcmp(d->prof_names[i], name) == 0)
      return i;
  }
  return kMaxProfKinds - 1;
}

struct ProfScope
{
  cudaEvent_t stop = nullptr;
  cudaStream_t st;
  ProfScope(rfm_decoder* d, ProfSlot* slots, const char* name, cudaStream_t stream) : st(stream)
  {
    if (!d->profiling)
      return;
    ProfSlot& sl = slots[ProfKind(d, name)];
    if (sl.used == sl.ev.size())
    {
      cudaEvent_t a, b;
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      sl.ev.emplace_back(a, b);
    }
    cudaEventRecord(sl.ev[sl.used].first, st);
    stop = sl.ev[sl.used].second;
    ++sl.used;
  }
  ~ProfScope()
  {
    if (stop)
      cudaEventRecord(stop, st);
  }
};
#define RFM_PROF(slots, name, stream, call)            \
  do                                                   \
  {                                                    \
    ProfScope ps_(d, slots, name, stream);             \
    call;                                              \
  } while (0)

void ProfCollect(rfm_decoder* d, ProfSlot* slots)
{
  static const bool timeline = RFM_KNOB("RFM_DEBUG_TIMELINE") != nullptr;
  for (int k = 0; k < kMaxProfKinds; ++k)
  {
    ProfSlot& sl = slots[k];
    for (size_t i = 0; i < sl.used; ++i)
    {
      float ms = 0.0f;
      if (cudaEventElapsedTime(&ms, sl.ev[i].first, sl.ev[i].second) == cudaSuccess)
      {
        d->prof_ms[k] += ms;
        d->prof_count[k] += 1;
        if (timeline && d->ev_base)
        {
          float t0 = 0.0f;
          if (cudaEventElapsedTime(&t0, d->ev_base, sl.ev[i].first) == cudaSuccess)
            fprintf(stderr, "TL %-16s %9.4f %9.4f\n", d->prof_names[k], t0, t0 + ms);
        }
      }
    }
    sl.used = 0;
  }
}

void ProfFree(ProfSlot* slots)
{
  for (int k = 0; k < kMaxProfKinds; ++k)
  {
    for (auto& e : slots[k].ev)
    {
      cudaEventDestroy(e.first);
      cudaEventDestroy(e.second);
    }
    slots[k].ev.clear();
    slots[k].used = 0;
  }
}

unsigned StageHist(const HalfBandStage& s) { return s.len == 3 ? 2u : (unsigned)s.len - 1; }

// cFmDecoder::Reset on the device state of one group (FmDecode.cpp:326-338 + RDSProcess.cpp:90-118)
cudaError_t ResetGroupState(rfm_decoder* d, Group& g, bool initial)
{
  const unsigned S = g.S;
  std::vector<float> st(g.state.n);
  cudaError_t e = cudaMemcpy(st.data(), g.state.p, st.size() * sizeof(float), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess)
    return e;
  auto zero = [&](int f) { std::fill(st.begin() + (size_t)f * S, st.begin() + (size_t)(f + 1) * S, 0.0f); };
  zero(SF_STEREO); zero(SF_STEREO1); zero(SF_STEREO2); zero(SF_IF_LEVEL); zero(SF_BB_MEAN); zero(SF_BB_LEVEL); zero(SF_DEMOD_DC);
  zero(SF_DEMOD_INCR); zero(SF_DEMOD_PHASE);
  zero(SF_RPLL_PHASE); zero(SF_RPLL_FREQ); zero(SF_RSYNC_W1); zero(SF_RSYNC_W2); zero(SF_RS_LASTSYNC);
  zero(SF_RS_LASTSLOPE); zero(SF_RS_LASTDATA); zero(SF_RS_LASTBIT);
  if (initial)
  {
    // cPilotPhaseLock ctor, FmDecode.cpp:131-139
    std::fill(st.begin() + (size_t)SF_PILOT_FREQ * S, st.begin() + (size_t)(SF_PILOT_FREQ + 1) * S, d->plan.pilot.freq0);
  }
  e = cudaMemcpy(g.state.p, st.data(), st.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e != cudaSuccess)
    return e;
  // InitLPFilter / InitConstFir clear the delay lines (FirFilter.cpp:138-144,313-319)
  // the LP delay line is the head of every stream's rlpV row
  {
    const unsigned lp_hist = (unsigned)d->plan.rlp_coef.size() - 1;
    e = cudaMemset2D(g.rlpV.p, (size_t)d->rlp_stride * sizeof(cf32), 0, (size_t)lp_hist * sizeof(cf32), S);
    if (e != cudaSuccess)
      return e;
  }
  return cudaMemset(g.mfV.p, 0, g.mfV.n * sizeof(float));
}

// Bring undrained slicer bits to the host and run the block-sync state machines on them.  All groups at once: the
// copies of every group are in flight together (pinned staging, each on the group's slicer stream), then ONE fan-out
// over the host cores covers all streams.
int DrainBits(rfm_decoder* d)
{
  if (d->pending_bits_bound == 0)
    return RFM_OK;
  const unsigned width = std::min(d->pending_bits_bound, d->bits_cap); // no stream can hold more undrained bits
  const size_t need = (size_t)d->S * (d->bits_cap + sizeof(unsigned)); // allocated once, at its largest
  if (d->h_drain_cap < need)
  {
    if (d->h_drain)
      cudaFreeHost(d->h_drain);
    d->h_drain = nullptr;
    d->h_drain_cap = 0;
    RFM_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&d->h_drain), need, cudaHostAllocDefault));
    d->h_drain_cap = need;
  }
  unsigned* h_counts = reinterpret_cast<unsigned*>(d->h_drain);
  uint8_t* h_bits = d->h_drain + (size_t)d->S * sizeof(unsigned);
  for (auto& g : d->groups)
  {
    RFM_CUDA(cudaMemcpyAsync(h_counts + g.s0, g.bit_count.p, g.S * sizeof(unsigned), cudaMemcpyDeviceToHost, g.sP));
    RFM_CUDA(cudaMemcpy2DAsync(h_bits + (size_t)g.s0 * width, width, g.bits.p, d->bits_cap, width, g.S,
                               cudaMemcpyDeviceToHost, g.sP));
    RFM_CUDA(cudaMemsetAsync(g.bit_count.p, 0, g.S * sizeof(unsigned), g.sP));
  }
  for (auto& g : d->groups)
    RFM_CUDA(cudaStreamSynchronize(g.sP));
  for (unsigned s = 0; s < d->S; ++s)
    if (h_counts[s] > width)
      return Fail(RFM_ERR_OVERFLOW, "RDS bit buffer overflow (internal drain bound violated)");
  // host block sync / FEC (RDSProcess.cpp:272-431) and group decoder: streams are independent
  auto work = [&](unsigned lo, unsigned hi) {
    for (unsigned s = lo; s < hi; ++s)
    {
      const uint8_t* b = h_bits + (size_t)s * width;
      const unsigned cnt = h_counts[s];
      if (cnt == 0)
        continue;
      auto& hb = d->host_bits[s];
      if (hb.size() + cnt > kMaxKeptBits) // raw bits are kept for rfm_decoder_rds_take_bits, bounded
        hb.erase(hb.begin(), hb.begin() + std::min(hb.size(), hb.size() + cnt - kMaxKeptBits));
      hb.insert(hb.end(), b, b + cnt);
      auto& sy = d->sync[s];
      const size_t had = sy.Groups().size();
      for (unsigned i = 0; i < cnt; ++i)
        sy.PushBit(b[i]);
      // RDSProcess.cpp:312,355: every decoded group goes straight to the group decoder
      auto& ud = d->uecp[s];
      for (size_t w = had; w + 4 <= sy.Groups().size(); w += 4)
        ud.Decode(sy.Groups().data() + w);
      // groups are kept for rfm_decoder_rds_take_groups, bounded like the raw bits (a caller that only reads the UECP
      // stream never takes them): the oldest go first
      auto& kept = sy.Groups();
      if (kept.size() > 4 * kMaxKeptGroups)
        kept.erase(kept.begin(), kept.begin() + (kept.size() - 4 * kMaxKeptGroups));
    }
  };
  const unsigned nthreads = std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), std::max(1u, d->S / 64));
  if (nthreads <= 1)
    work(0, d->S);
  else
  {
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nthreads; ++t)
      pool.emplace_back(work, (unsigned)((uint64_t)d->S * t / nthreads), (unsigned)((uint64_t)d->S * (t + 1) / nthreads));
    work(0, (unsigned)((uint64_t)d->S / nthreads));
    for (auto& th : pool)
      th.join();
  }
  d->pending_bits_bound = 0;
  return RFM_OK;
}

struct BlockGeom
{
  unsigned n, nb, na, nr;
  unsigned hb_n[kMaxDecStages + 1]; // samples entering stage k; hb_n[nstages] == nr
  unsigned short_mask;              // stage k received fewer samples than its FIR is long (DownConvert.cpp:519-520)
  bool rds_skip;                    // the RDS branch does not run for this block (see PlanBlock)
  float a_pos_next;
  unsigned in_pos_next;
};

// Sample counts of one block.  The audio path takes ANY n (>= the input FIR order).  The RDS decimate-by-2 chain
// follows the reference for counts it was not written for (DownConvert.cpp:498-550, pinned against the compiled
// reference in tests/test_gpu_parity.py::test_default_rtlsdr_block_at_1200k): a generic half-band stage fed an ODD
// count m makes (m + 1) / 2 outputs (its loop runs i = 0, 2, .. < m; the last output ends on the newest sample) and
// restarts its decimation phase at the next block's first sample; fed FEWER samples than it has taps it returns the
// first m / 2 inputs unfiltered and keeps its delay line.  Only the fixed 11-tap and CIC3 stages (rates below
// ~480 kS/s) read outside their input for odd / short counts in the reference -- undefined there, so such a block
// skips the RDS branch here (no bits, RDS state untouched) while its audio is produced as usual.
int PlanBlock(const rfm_decoder* d, unsigned n, BlockGeom* g)
{
  const DecoderPlan& p = d->plan;
  g->n = n;
  const unsigned ds = p.downsample;
  // integer decimator, DownConvert.cpp:105-132
  unsigned pos = d->in_pos;
  g->nb = (pos < n) ? (n - pos + ds - 1) / ds : 0;
  g->in_pos_next = pos + g->nb * ds - n;
  g->na = FractionalOutputs(d->a_pos, p.a_pstep, g->nb, &g->a_pos_next);
  g->short_mask = 0;
  g->rds_skip = false;
  unsigned m = g->nb;
  for (size_t k = 0; k < p.rds_stages.size(); ++k)
  {
    g->hb_n[k] = m;
    const HalfBandStage& hs = p.rds_stages[k];
    const bool generic = hs.len != 3 && !hs.fixed11;
    if (generic)
    {
      if (m < (unsigned)hs.len)
      {
        g->short_mask |= 1u << k;
        m /= 2;
      }
      else
        m = (m + 1) / 2;
    }
    else
    {
      if (m % 2 != 0 || m < 18)
        g->rds_skip = true;
      m /= 2;
    }
  }
  g->hb_n[p.rds_stages.size()] = m;
  g->nr = m;
  if (g->rds_skip)
    g->nr = 0;
  return RFM_OK;
}

// timing experiments only (results are wrong when a stage is skipped): RFM_DEBUG_SKIP=front,lanes,rest
bool DebugSkip(const char* what)
{
  static const char* env = RFM_KNOB("RFM_DEBUG_SKIP");
  return env && strstr(env, what);
}

// Stage F of one block for one group (stream sF): IF meter, front end.
void EnqueueStageF(rfm_decoder* d, Group& g, const void* d_in, size_t in_stride, IqFormat fmt, const BlockGeom& bg,
                   unsigned par)
{
  const DecoderPlan& p = d->plan;
  cudaStream_t st = g.sF;
  const unsigned S = g.S;

  FrontParams fp;
  fp.in = d_in; fp.in_stride = in_stride; fp.n = bg.n; fp.S = S; fp.order = p.in_order; fp.ds = p.downsample;
  fp.p0 = d->in_pos; fp.nout = bg.nb; fp.idx0 = d->tuner_idx; fp.lut = d->d_lut.p; fp.tuner = d->d_tuner.p;
  fp.coeff = d->d_in_coeff.p; fp.coeff_host = p.in_coeff.data(); fp.tail = g.tail.p; fp.z = g.z[par].p; fp.z_stride = d->z_stride;
  fp.sm_count = d->part.rest ? d->part.rest_sms : 0;
  fp.fused = d->cfg.fir_fused != 0;
  RFM_PROF(g.prof, "k_if_level", st, launch_if_level(fp, g.state.p, fmt, st));
  RFM_PROF(g.prof, "k_front", st, launch_front(fp, fmt, st));
  RFM_PROF(g.prof, "k_front_tail", st, launch_front_tail(fp, fmt, st));

  // FM-demodulator PLL, time-parallel (throughput work like the front end).  It overwrites incr[par], which the
  // lanes of block k-2 were reading.
  cudaStreamWaitEvent(st, g.ev_lanes[par], 0);
  DemodSpecParams dp;
  dp.z = g.z[par].p; dp.z_stride = d->z_stride; dp.nb = bg.nb; dp.S = S; dp.state = g.state.p;
  dp.warm = p.fs_bb < 225000.0f ? 96u : 160u; // measured miss rates: DESIGN.md 3.1
  dp.demod = {p.demod_gain, p.nco_lo, p.nco_hi, p.pll_alpha, p.pll_beta};
  dp.incr = g.incr[par].p; dp.w_stride = d->z_stride; dp.st_start = g.dm_start.p; dp.st_end = g.dm_end.p;
  dp.repairs = d->d_repairs.p;
  RFM_PROF(g.prof, "k_demod_spec", st, launch_demod_spec(dp, st));
  RFM_PROF(g.prof, "k_demod_fix", st, launch_demod_fix(dp, st));
  g_launches += 7;
}

// Stage A of one block for one group (stream sA): history hand-over, PLL lanes.
void EnqueueStageA(rfm_decoder* d, Group& g, const BlockGeom& bg, unsigned par, unsigned par3)
{
  const DecoderPlan& p = d->plan;
  cudaStream_t st = g.sA;
  const unsigned S = g.S;
  const unsigned a_hist = p.a_order;

  // history of the baseband / L-R rows: last a_hist samples of the previous block (other parity) -> head of this one
  TailParams tp;
  tp.count = 2;
  const unsigned prev3 = (par3 + 2u) % 3u;
  tp.d[0] = {g.bbV[prev3].p, g.bbV[par3].p, d->a_stride * sizeof(float), a_hist, d->last_nb, 4, S};
  tp.d[1] = {g.rawV[prev3].p, g.rawV[par3].p, d->a_stride * sizeof(float), a_hist, d->last_nb, 4, S};
  RFM_PROF(g.prof, "k_tails", st, launch_tails(tp, S, st));

  LanesParams lp;
  lp.incr = g.incr[par].p; lp.w_stride = d->z_stride; lp.nb = bg.nb; lp.S = S; lp.state = g.state.p;
  lp.demod = {p.demod_gain, p.nco_lo, p.nco_hi, p.pll_alpha, p.pll_beta};
  lp.pilot = {p.pilot.minfreq, p.pilot.maxfreq, p.pilot.b0, p.pilot.a1, p.pilot.a2, p.pilot.lb0, p.pilot.lb1,
              p.pilot.minsignal, p.pilot.lock_delay};
  lp.bbV = g.bbV[par3].p; lp.rawV = g.rawV[par3].p; lp.a_stride = d->a_stride; lp.a_hist = a_hist; lp.parity = par3;
  lp.packed = d->part.lanes != nullptr; // few SMs for all lanes CTAs: the form that fits 12 of them on one SM
  RFM_PROF(g.prof, "k_bb_lanes", st, launch_bb_lanes(lp, st));
  g_launches += 2;
}

// Stage B of one block for one group, four streams:
//   sB  resamplers (bbV / rawV [par3] -> lpS / lpM [par])           sC  audio LP, deemphasis, notch, matrix (-> audio)
//   sR  RDS front (bbV [par3], oscV [par3] -> rlp_out [par])        sP  Costas loop, matched filter, slicer (-> bits)
// The lane kernels (k_rds_pll, k_audio_tail, k_rds_slice) are latency-bound and stretch when they share the SMs with
// the FIR kernels; on their own streams they overlap the FIR kernels of the NEXT block instead of delaying them.
void EnqueueStageB(rfm_decoder* d, Group& g, const BlockGeom& bg, unsigned par, unsigned par3, float* d_audio,
                   size_t audio_stride)
{
  const DecoderPlan& p = d->plan;
  const unsigned S = g.S;
  const unsigned a_hist = p.a_order;
  const unsigned lp_taps = (unsigned)p.lp_coef.size(), rlp_taps = (unsigned)p.rlp_coef.size();
  const unsigned mf_taps = (unsigned)p.mf_coef.size();
  const unsigned nst = (unsigned)p.rds_stages.size();

  // ---- sB: fractional resamplers
  cudaStream_t st = g.sB;
  ResampleParams rp;
  rp.bbV = g.bbV[par3].p; rp.rawV = g.rawV[par3].p; rp.a_stride = d->a_stride; rp.order = p.a_order; rp.nb = bg.nb;
  rp.S = S; rp.na = bg.na; rp.pos_frac = d->a_pos; rp.pstep = p.a_pstep; rp.coeff = d->d_a_coeff.p;
  rp.lpS = g.lpS[par].p; rp.lpM = g.lpM[par].p; rp.lp_stride = d->lp_stride; rp.lp_hist = lp_taps - 1;
  rp.kk = d->res_kk[par3].p; rp.meta = d->res_meta[par3].p; rp.lp = d->res_lp;
  rp.fused = d->cfg.fir_fused != 0;
  RFM_PROF(g.prof, "k_resample", st, launch_resample_tiled(rp, st));
  cudaEventRecord(g.ev_res[par], st);
  ++g_launches;

  // ---- sC: audio tail.  History of the LP input rows: last lp_taps-1 samples of the previous block (other parity)
  st = g.sC;
  cudaStreamWaitEvent(st, g.ev_res[par], 0);
  {
    TailParams tpa;
    tpa.count = 2;
    tpa.d[0] = {g.lpS[par ^ 1u].p, g.lpS[par].p, d->lp_stride * sizeof(float), lp_taps - 1, d->last_na, 4, S};
    tpa.d[1] = {g.lpM[par ^ 1u].p, g.lpM[par].p, d->lp_stride * sizeof(float), lp_taps - 1, d->last_na, 4, S};
    RFM_PROF(g.prof, "k_tails", st, launch_tails(tpa, S, st));
    cudaEventRecord(g.ev_carry[par], st);
  }
  RotFirParams f29;
  f29.inA = g.lpS[par].p; f29.inB = g.lpM[par].p; f29.in_stride = d->lp_stride; f29.outA = g.fS.p; f29.outB = g.fM.p;
  f29.out_stride = d->na_max; f29.out_off = 0; f29.n = bg.na; f29.S = S; f29.taps = lp_taps; f29.g0 = d->lp_g;
  f29.coef = d->d_lp_coef.p; f29.cplx = 0; f29.fused = d->cfg.fir_fused != 0;
  RFM_PROF(g.prof, "k_rotfir_lp29", st, launch_rotfir(f29, st));

  AudioTailParams at;
  at.inS = g.fS.p; at.inM = g.fM.p; at.in_stride = d->na_max; at.na = bg.na; at.S = S; at.state = g.state.p;
  at.de_alpha = p.de_alpha; at.notch = {p.notch.A1, p.notch.A2, p.notch.B0, p.notch.B1, p.notch.B2};
  at.audio = d_audio; at.audio_stride = audio_stride; at.parity = par3;
  RFM_PROF(g.prof, "k_audio_tail", st, launch_audio_tail(at, st));
  g_launches += 3;

  // ---- sR: RDS front (mix, decimate-by-2 chain, LP)
  st = g.sR;
  if (!bg.rds_skip)
  {
  RdsFrontParams rf;
  memset(&rf, 0, sizeof(rf));
  rf.bbV = g.bbV[par3].p; rf.a_stride = d->a_stride; rf.a_hist = a_hist;
  rf.osc = d->oscV[par3].p + d->osc_hist; rf.nb = bg.nb; rf.S = S; rf.nst = nst;
  for (unsigned k = 0; k < nst; ++k)
  {
    const HalfBandStage& hs = p.rds_stages[k];
    rf.st[k].kind = hs.len == 3 ? 2 : (hs.fixed11 ? 1 : 0);
    rf.st[k].len = (unsigned)hs.len;
    rf.st[k].hist = StageHist(hs);
    rf.st[k].h = hs.h ? d->d_hb[k].p : nullptr;
    rf.st[k].h_host = hs.h;
    rf.tail_off[k] = d->rds_tail_off[k];
  }
  rf.tail_off[nst] = d->rds_tail_off[nst];
  rf.lp_coef = d->d_rlp_coef.p; rf.lp_n = rlp_taps; rf.g0 = d->rlp_g;
  rf.tails = g.rds_tails.p; rf.tail_stride = d->rds_tail_stride;
  rf.out = nullptr; rf.dec_out = nullptr; rf.out_stride = d->nr_stride;
  rf.lp_v = g.rlpV.p; rf.lp_v_stride = d->rlp_stride; // decimator output -> [LP history | block] rows
  rf.short_mask = bg.short_mask;
  RFM_PROF(g.prof, "k_rds_front", st, launch_rds_front(rf, st));
  {
    // the 2.4 kHz LP (RDSProcess.cpp:128), lane = stream form, then its history carry
    RotFirParams flp;
    flp.inA = reinterpret_cast<const float*>(g.rlpV.p); flp.inB = nullptr; flp.in_stride = d->rlp_stride;
    flp.outA = reinterpret_cast<float*>(g.rlp_out[par].p); flp.outB = nullptr; flp.out_stride = d->nr_stride;
    flp.out_off = 0; flp.n = bg.nr; flp.S = S; flp.taps = rlp_taps; flp.g0 = d->rlp_g; flp.coef = d->d_rlp_coef.p;
    flp.cplx = 1; flp.fused = d->cfg.fir_fused != 0;
    RFM_PROF(g.prof, "k_rotfir_rdslp", st, launch_rotfir(flp, st));
    TailParams tpl;
    tpl.count = 1;
    tpl.d[0] = {g.rlpV.p, g.rlpV.p, d->rlp_stride * sizeof(cf32), rlp_taps - 1, bg.nr, 8, S};
    RFM_PROF(g.prof, "k_tails", st, launch_tails(tpl, S, st));
  }
  }
  cudaEventRecord(g.ev_rds[par3], st);
  g_launches += 3;

  // ---- sP: Costas loop, matched filter, bit clock + slicer
  st = g.sP;
  cudaStreamWaitEvent(st, g.ev_rds[par3], 0);
  if (bg.rds_skip)
    return;
  RdsPllParams pp;
  pp.in = g.rlp_out[par].p; pp.in_stride = d->nr_stride; pp.nr = bg.nr; pp.S = S; pp.state = g.state.p;
  pp.lo = p.rpll_lo; pp.hi = p.rpll_hi; pp.alpha = p.rpll_alpha; pp.beta = p.rpll_beta;
  pp.out = g.mfV.p; pp.out_stride = d->mf_stride; pp.out_off = mf_taps - 1;
  RFM_PROF(g.prof, "k_rds_pll", st, launch_rds_pll(pp, st));

  RotFirParams fmf;
  fmf.inA = g.mfV.p; fmf.inB = nullptr; fmf.in_stride = d->mf_stride; fmf.outA = g.mf_out.p; fmf.outB = nullptr;
  fmf.out_stride = d->nr_stride; fmf.out_off = 0; fmf.n = bg.nr; fmf.S = S; fmf.taps = mf_taps; fmf.g0 = d->mf_g;
  fmf.coef = d->d_mf_coef.p; fmf.cplx = 0; fmf.fused = d->cfg.fir_fused != 0;
  RFM_PROF(g.prof, "k_rotfir_rdsmf", st, launch_rotfir(fmf, st));

  RdsSliceParams sp;
  sp.in = g.mf_out.p; sp.in_stride = d->nr_stride; sp.nr = bg.nr; sp.S = S; sp.state = g.state.p;
  sp.sync = {p.rsync.A1, p.rsync.A2, p.rsync.B0, p.rsync.B1, p.rsync.B2};
  sp.bits = g.bits.p; sp.bits_cap = d->bits_cap; sp.bit_count = g.bit_count.p;
  RFM_PROF(g.prof, "k_rds_slice", st, launch_rds_slice(sp, st));
  g_launches += 3;

  // in-place history carry of the matched filter's input rows
  TailParams tp;
  tp.count = 0;
  if (mf_taps > 1)
    tp.d[tp.count++] = {g.mfV.p, g.mfV.p, d->mf_stride * sizeof(float), mf_taps - 1, bg.nr, 4, S};
  RFM_PROF(g.prof, "k_tails", st, launch_tails(tp, S, st));
  ++g_launches;
}

// One block for all groups.  Inputs / outputs are device pointers for the whole batch (host pointers when
// host_staged).  Work is only enqueued; the device entry points return without waiting (rfm_decoder_wait).
int ProcessDevice(rfm_decoder* d, const void* d_in, size_t in_stride, IqFormat fmt, unsigned n, float* d_audio,
                  size_t audio_stride, uint32_t* n_audio_floats, cudaStream_t user, bool host_staged,
                  bool host_sync = true)
{
  if (n == 0)
  {
    if (n_audio_floats)
      *n_audio_floats = 0;
    return RFM_OK;
  }
  if (n > d->maxn)
    return Fail(RFM_ERR_INVALID, "n exceeds max_block_len");
  if (n < d->plan.in_order)
    return Fail(RFM_ERR_UNSUPPORTED, "blocks shorter than the input FIR order (8*downsample) are not supported");
  BlockGeom bg;
  int rc = PlanBlock(d, n, &bg);
  if (rc != RFM_OK)
    return rc;
  if (2 * (size_t)bg.na > audio_stride)
    return Fail(RFM_ERR_OVERFLOW, "audio_stride smaller than the floats produced per stream");
  if (!host_staged && ((audio_stride & 1u) || (reinterpret_cast<uintptr_t>(d_audio) & 7u)))
    return Fail(RFM_ERR_INVALID, "device audio rows must be 8-byte aligned (even audio_stride): L,R pairs are stored as float2");
  RFM_CUDA(cudaSetDevice(d->device));

  // drain the RDS bit buffers before they could overflow
  const unsigned worst_bits = bg.nr / 8 + 4; // >= 8 samples per bit at every supported rate; overflow is checked
  if (d->pending_bits_bound + worst_bits > d->bits_cap)
  {
    rc = DrainBits(d);
    if (rc != RFM_OK)
      return rc;
  }

  const unsigned par = (unsigned)(d->block_index & 1u);  // z / incr (front -> demodulator -> lanes)
  const unsigned par3 = (unsigned)(d->block_index % 3u); // everything handed to stage B
  const unsigned prev3 = (par3 + 2u) % 3u;
  if (!host_staged)
    RFM_CUDA(cudaEventRecord(d->ev_fork, user)); // stage A must see what is already enqueued on the caller's stream

  // NCO oscillator table of this block (shared by all streams), on its own stream: it only depends on the
  // sample count, so it runs ahead of the data.
  for (auto& g : d->groups)
    RFM_CUDA(cudaStreamWaitEvent(d->s_osc, g.ev_rest[par3], 0)); // readers of oscV[par3] three blocks ago
  {
    TailParams tp;
    tp.count = 1;
    tp.d[0] = {d->oscV[prev3].p, d->oscV[par3].p, 0, d->osc_hist, d->last_nb_rds, 8, 1};
    RFM_PROF(d->main_prof, "k_tails", d->s_osc, launch_tails(tp, 1, d->s_osc));
    OscParams op;
    op.oscV = d->oscV[par3].p; op.osc_hist = d->osc_hist; op.nb = bg.rds_skip ? 0u : bg.nb; op.osc1 = d->osc1.p;
    op.cosv = d->plan.rds_osc.cosv; op.sinv = d->plan.rds_osc.sinv;
    RFM_PROF(d->main_prof, "k_osc", d->s_osc, launch_osc(op, d->s_osc));
    ResTapsParams tp2;
    tp2.pos_frac = d->a_pos; tp2.pstep = d->plan.a_pstep; tp2.na = bg.na; tp2.order = d->plan.a_order;
    tp2.lp = d->res_lp; tp2.coeff = d->d_a_coeff.p; tp2.kk = d->res_kk[par3].p; tp2.meta = d->res_meta[par3].p;
    RFM_PROF(d->main_prof, "k_res_taps", d->s_osc, launch_res_taps(tp2, d->s_osc));
    g_launches += 3;
    RFM_CUDA(cudaEventRecord(d->ev_osc[par3], d->s_osc));
  }

  const size_t esz = IqBytes(fmt);
  for (auto& g : d->groups)
  {
    const unsigned char* in_g = reinterpret_cast<const unsigned char*>(d_in) + (size_t)g.s0 * in_stride * esz;
    float* audio_g = d_audio + (size_t)g.s0 * audio_stride;
    const void* in_dev = in_g;
    float* audio_dev = audio_g;
    size_t in_stride_dev = in_stride, audio_stride_dev = audio_stride;
    // ---- stage F
    if (!host_staged)
      RFM_CUDA(cudaStreamWaitEvent(g.sF, d->ev_fork, 0));
    // (z[par] was last read by the demodulator of block k-2, on this same stream)
    if (host_staged)
    {
      // one contiguous copy when the caller's rows are dense (the usual case): the staging rows are then packed too
      if (in_stride == n)
      {
        {
          ProfScope ps_(d, g.prof, "copy_h2d", g.sF);
          RFM_CUDA(cudaMemcpyAsync(g.in_stage.p, in_g, (size_t)g.S * n * esz, cudaMemcpyHostToDevice, g.sF));
        }
        in_stride_dev = n;
      }
      else
      {
        RFM_CUDA(cudaMemcpy2DAsync(g.in_stage.p, (size_t)d->maxn * esz, in_g, in_stride * esz, (size_t)n * esz, g.S,
                                   cudaMemcpyHostToDevice, g.sF));
        in_stride_dev = d->maxn;
      }
      in_dev = g.in_stage.p;
      audio_dev = g.audio_stage.p;
      audio_stride_dev = d->audio_cap;
    }
    if (!DebugSkip("front"))
      EnqueueStageF(d, g, in_dev, in_stride_dev, fmt, bg, par);
    RFM_CUDA(cudaEventRecord(g.ev_front[par], g.sF));
    // ---- stage A
    RFM_CUDA(cudaStreamWaitEvent(g.sA, g.ev_front[par], 0));
    RFM_CUDA(cudaStreamWaitEvent(g.sA, g.ev_rest[par3], 0)); // stage B of block k-3 has released bbV / rawV [par3]
    RFM_CUDA(cudaStreamWaitEvent(g.sA, g.ev_aud[par3], 0));   // ... and its audio tail the stereo-flag slot (k mod 3).  Waiting
                                                              // for block k-2's instead made lanes(k) -> resamplers(k) -> audio
                                                              // tail(k) -> lanes(k+2) a two-step cycle that bound the step
    if (!DebugSkip("lanes"))
      EnqueueStageA(d, g, bg, par, par3);
    RFM_CUDA(cudaEventRecord(g.ev_lanes[par], g.sA));
    // ---- stage B
    for (cudaStream_t st : {g.sB, g.sR})
    {
      RFM_CUDA(cudaStreamWaitEvent(st, g.ev_lanes[par], 0));
      RFM_CUDA(cudaStreamWaitEvent(st, d->ev_osc[par3], 0));
    }
    // lpS / lpM [par]: the audio tail of block k-2 has read them and block k-1 has carried its history out of them
    // (both on sC, in that order)
    RFM_CUDA(cudaStreamWaitEvent(g.sB, g.ev_carry[par ^ 1u], 0));
    RFM_CUDA(cudaStreamWaitEvent(g.sR, g.ev_pll[par], 0)); // RDS PLL of block k-2 has released rlp_out [par]
    if (!DebugSkip("rest"))
      EnqueueStageB(d, g, bg, par, par3, audio_dev, audio_stride_dev);
    RFM_CUDA(cudaStreamWaitEvent(g.sB, g.ev_rds[par3], 0)); // ev_rest: both readers of bbV / rawV / oscV [par3] are done
    RFM_CUDA(cudaEventRecord(g.ev_rest[par3], g.sB));
    RFM_CUDA(cudaEventRecord(g.ev_pll[par], g.sP));
    if (host_staged)
    {
      ProfScope ps_(d, g.prof, "copy_d2h", g.sC);
      RFM_CUDA(cudaMemcpy2DAsync(audio_g, audio_stride * sizeof(float), g.audio_stage.p,
                                 (size_t)d->audio_cap * sizeof(float), (size_t)2 * bg.na * sizeof(float), g.S,
                                 cudaMemcpyDeviceToHost, g.sC));
    }
    RFM_CUDA(cudaEventRecord(g.ev_aud[par3], g.sC));
  }
  RFM_CUDA(cudaGetLastError());

  // advance the lock-step state
  d->tuner_idx = (d->tuner_idx + n) % kTunerTable;
  d->in_pos = bg.in_pos_next;
  d->a_pos = bg.a_pos_next;
  d->lp_g = (d->lp_g + bg.na) % (unsigned)d->plan.lp_coef.size();
  d->rlp_g = (d->rlp_g + bg.nr) % (unsigned)d->plan.rlp_coef.size();
  d->mf_g = (d->mf_g + bg.nr) % (unsigned)d->plan.mf_coef.size();
  d->pending_bits_bound += worst_bits;
  d->last_n = n; d->last_nb = bg.nb; d->last_na = bg.na; d->last_nr = bg.nr;
  d->last_nb_rds = bg.rds_skip ? 0u : bg.nb;
  memcpy(d->last_hb_n, bg.hb_n, sizeof(bg.hb_n));
  d->block_index += 1;
  if (n_audio_floats)
    *n_audio_floats = 2 * bg.na;
  if (host_staged && host_sync)
    for (auto& g : d->groups)
      RFM_CUDA(cudaStreamSynchronize(g.sC)); // the audio is on the host (the RDS branch may still be running: the
                                             // rds_take_* entry points synchronise it)
  return RFM_OK;
}

Group* FindGroup(rfm_decoder* d, unsigned stream, unsigned* local)
{
  for (auto& g : d->groups)
    if (stream >= g.s0 && stream < g.s0 + g.S)
    {
      *local = stream - g.s0;
      return &g;
    }
  return nullptr;
}

int SyncAll(rfm_decoder* d)
{
  RFM_CUDA(cudaSetDevice(d->device));
  for (auto& g : d->groups)
  {
    cudaStream_t all[6];
    g.AllStreams(all);
    for (cudaStream_t st : all)
      if (st)
        RFM_CUDA(cudaStreamSynchronize(st));
  }
  RFM_CUDA(cudaStreamSynchronize(d->s_osc));
  return RFM_OK;
}

} // namespace

extern "C"
{

const char* rfm_last_error(void) { return g_err.c_str(); }
const char* rfm_version(void) { return "radiofm_b200 0.2 (sm_100a)"; }

uint32_t rfm_iq_format_bytes(int format)
{
  return (format >= RFM_IQ_U8 && format <= RFM_IQ_CF32) ? IqBytes(format) : 0u;
}
uint64_t rfm_launch_count(void) { return g_launches.load(); }

void rfm_config_default(rfm_config* c)
{
  memset(c, 0, sizeof(*c));
  c->sample_rate_if = 1.0e6;       // RadioReceiver.cpp:184
  c->tuning_offset = -0.15e6;      // RadioReceiver.cpp:237,297
  c->sample_rate_pcm = 48000.0;    // OUTPUT_SAMPLERATE
  c->bandwidth_pcm = 15000.0;
  c->downsample = 4;               // RadioReceiver.cpp:285
  c->us_deemphasis = 0;
  c->n_streams = 1;
  c->max_block_len = 65536;        // cRtlSdrSource::default_block_length
  c->device = -1;
  c->n_groups = 0;
  c->lanes_sms = 0;
  c->fir_fused = 0;
}

int rfm_decoder_create(const rfm_config* cfg, rfm_decoder** out)
{
  if (!cfg || !out)
    return Fail(RFM_ERR_INVALID, "null argument");
  *out = nullptr;
  if (cfg->n_streams == 0 || cfg->downsample == 0 || cfg->max_block_len == 0 || cfg->sample_rate_if <= 0 ||
      cfg->sample_rate_pcm <= 0)
    return Fail(RFM_ERR_INVALID, "invalid configuration");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return Fail(RFM_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  int dev = cfg->device;
  if (dev < 0)
    RFM_CUDA(cudaGetDevice(&dev));
  if (dev >= ndev)
    return Fail(RFM_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  RFM_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    return Fail(RFM_ERR_NO_DEVICE, std::string("kernels are built for sm_100a only; device is ") + prop.name);
  RFM_CUDA(cudaSetDevice(dev));

  rfm_decoder* d = new rfm_decoder;
  d->cfg = *cfg;
  d->device = dev;
  d->S = cfg->n_streams;
  d->maxn = cfg->max_block_len;
  d->plan = PlanDecoder(cfg->sample_rate_if, cfg->tuning_offset, cfg->sample_rate_pcm, cfg->bandwidth_pcm,
                        cfg->downsample, cfg->us_deemphasis != 0);
  const DecoderPlan& p = d->plan;
  auto bail = [&](int code, const std::string& m) {
    FreeDecoder(d);
    return Fail(code, m);
  };
  if (p.rds_stages.empty() || p.rds_stages.size() > kRfMaxStages)
    return bail(RFM_ERR_UNSUPPORTED, "baseband rate outside the supported range (RDS decimation chain empty)");
  if (p.a_order > 512 || p.in_order > 512 || p.a_order < 2)
    return bail(RFM_ERR_UNSUPPORTED, "filter order outside the supported range (<= 512)");
  if (p.mf_coef.size() < 2 || p.rlp_coef.size() > kMaxFirTapsDev)
    return bail(RFM_ERR_UNSUPPORTED, "RDS filter length outside the supported range");

  const unsigned ds = p.downsample;
  d->nb_max = (d->maxn + ds - 1) / ds + 1;
  d->na_max = (unsigned)(d->nb_max / p.a_ratio) + 4;
  d->nr_max = d->nb_max; // generous: halved per stage below
  d->z_stride = AlignUp(d->nb_max, 16);
  d->a_stride = AlignUp(p.a_order + d->nb_max + 4, 32); // + 4: the resampler's 16-byte tile copies may end past the block
  d->lp_stride = AlignUp((unsigned)p.lp_coef.size() - 1 + d->na_max, 32);
  unsigned m = d->nb_max;
  for (size_t k = 0; k < p.rds_stages.size(); ++k)
  {
    d->hb_stride[k] = AlignUp(StageHist(p.rds_stages[k]) + m, 16);
    m = m / 2 + 1;
  }
  d->nr_max = m;
  d->nr_stride = AlignUp(d->nr_max, 16);
  d->rlp_stride = AlignUp((unsigned)p.rlp_coef.size() - 1 + d->nr_max, 16);
  d->mf_stride = AlignUp((unsigned)p.mf_coef.size() - 1 + d->nr_max, 32);
  d->osc_hist = StageHist(p.rds_stages[0]);
  {
    unsigned off = 0;
    for (size_t k = 0; k < p.rds_stages.size(); ++k)
    {
      d->rds_tail_off[k] = off;
      off += StageHist(p.rds_stages[k]);
    }
    d->rds_tail_off[p.rds_stages.size()] = off;
    off += (unsigned)p.rlp_coef.size() - 1;
    d->rds_tail_stride = AlignUp(off, 4);
  }
  d->bits_cap = 4096;
  d->audio_cap = AlignUp(2 * d->na_max, 32);

#define RFM_TRY(expr)                                                                                    \
  do                                                                                                     \
  {                                                                                                      \
    cudaError_t e_ = (expr);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return bail(RFM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));                    \
  } while (0)

  RFM_TRY(Upload(d->d_lut, p.u8lut, 256));
  RFM_TRY(Upload(d->d_tuner, p.tuner, 2 * kTunerTable));
  RFM_TRY(Upload(d->d_in_coeff, p.in_coeff.data(), p.in_coeff.size()));
  RFM_TRY(Upload(d->d_a_coeff, p.a_coeff.data(), p.a_coeff.size()));
  RFM_TRY(Upload(d->d_lp_coef, p.lp_coef.data(), p.lp_coef.size()));
  RFM_TRY(Upload(d->d_rlp_coef, p.rlp_coef.data(), p.rlp_coef.size()));
  RFM_TRY(Upload(d->d_mf_coef, p.mf_coef.data(), p.mf_coef.size()));
  for (size_t k = 0; k < p.rds_stages.size(); ++k)
  {
    if (p.rds_stages[k].h)
      RFM_TRY(Upload(d->d_hb[k], p.rds_stages[k].h, (size_t)p.rds_stages[k].len));
    else
      RFM_TRY(d->d_hb[k].Alloc(4));
  }
  RFM_TRY(d->d_repairs.Alloc(1));
  // time steps per group of 4 outputs: one window + 3 output spacings, + the alignment of both ends to 4 samples
  d->res_lp = AlignUp(p.a_order + 1 + 3 * ((unsigned)p.a_ratio + 1) + 4 + 6, 4);
  for (int b = 0; b < 3; ++b)
  {
    RFM_TRY(d->res_kk[b].Alloc((size_t)(d->na_max / 4 + 2) * d->res_lp * 4));
    RFM_TRY(d->res_meta[b].Alloc((size_t)(d->na_max / 4 + 2) * 2));
  }
  for (int b = 0; b < 3; ++b)
    RFM_TRY(d->oscV[b].Alloc((size_t)d->osc_hist + d->nb_max));
  {
    const float one[2] = {1.0f, 0.0f}; // m_Osc1 initial unit vector, DownConvert.cpp:283-284
    RFM_TRY(Upload(d->osc1, one, 2));
  }
  {
    // SM partition (rfm_config::lanes_sms; RFM_LANES_SMS overrides it in the experiments build)
    unsigned n = cfg->lanes_sms;
    if (n == 0) // automatic: a batch wide enough that the FIR kernels fill the device (measured: DESIGN.md section 4)
      n = (cfg->n_streams >= 2048 && prop.multiProcessorCount >= 100) ? 24u : 0u;
    if (const char* e = RFM_KNOB("RFM_LANES_SMS"))
      n = (unsigned)KnobInt(e, 0);
    if (n >= 8)
    {
      std::string why;
      if (!MakeSmPartition(d->device, n, &d->part, &why))
      {
        FreeSmPartition(&d->part);
        SetLastError("lanes_sms ignored: " + why); // creation still succeeds, on ordinary streams
      }
      else if (RFM_KNOB("RFM_DEBUG_TIMELINE"))
        fprintf(stderr, "radiofm_b200: lanes on %u SMs, everything else on %u\n", d->part.lanes_sms, d->part.rest_sms);
    }
  }
  // which streams live in the lanes partition: letters of RFM_LANES_STREAMS among A (lanes), O (oscillator / resampler
  // tables), P (RDS PLL, matched filter, slicer), C (audio tail), R (RDS front), B (resamplers), F (front end)
  const char* in_lanes = RFM_KNOB("RFM_LANES_STREAMS") ? RFM_KNOB("RFM_LANES_STREAMS") : "AO";
  auto ctx_of = [&](char which) { return strchr(in_lanes, which) ? d->part.lanes : d->part.rest; };
  {
    int lo = 0, hi = 0;
    RFM_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    RFM_TRY(MakeStream(ctx_of('O'), &d->s_osc, lo));
  }
  RFM_TRY(cudaEventCreateWithFlags(&d->ev_fork, cudaEventDisableTiming));
  for (int b = 0; b < 3; ++b)
    RFM_TRY(cudaEventCreateWithFlags(&d->ev_osc[b], cudaEventDisableTiming));
  RFM_TRY(cudaEventCreateWithFlags(&d->ev_join, cudaEventDisableTiming));

  unsigned G = cfg->n_groups;
  if (G == 0)
    G = 1;
  G = std::min(G, d->S);
  d->groups.resize(G);
  const size_t esz_max = 8; // cf32 input
  for (unsigned gi = 0; gi < G; ++gi)
  {
    Group& g = d->groups[gi];
    g.s0 = (unsigned)((uint64_t)d->S * gi / G);
    g.S = (unsigned)((uint64_t)d->S * (gi + 1) / G) - g.s0;
    const size_t S = g.S;
    {
      int prio_lo = 0, prio_hi = 0; // the latency-bound lanes kernel gets its CTAs placed first
      RFM_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
      if (RFM_KNOB("RFM_DEBUG_NOPRIO"))
        prio_hi = prio_lo;
      // sA (demodulator + lanes) is the critical chain, the front end feeds it; the audio / RDS branches have slack
      const char* flow = RFM_KNOB("RFM_DEBUG_FLOW");
      const int mode = KnobInt(flow, 0);
      // (stage B one step above the lowest priority: the lowest is left to the companion stream, whose long-running
      // front-end CTAs otherwise keep the small stage-B kernels of a narrow batch waiting for an SM slot for milliseconds)
      int pA = prio_hi, pF = std::min(prio_lo, prio_hi + 1), pB = (prio_lo - 1 > prio_hi + 1) ? prio_lo - 1 : prio_lo;
      int pL = KnobInt(RFM_KNOB("RFM_DEBUG_LANEPRIO"), 0) + prio_hi; // small lane kernels of stage B
      if (mode == 1) { pF = prio_lo; }
      if (mode == 2) { pF = prio_lo; pB = std::min(prio_lo, prio_hi + 1); }
      if (mode == 3) { pA = prio_lo; pF = prio_lo; pB = prio_hi; }
      RFM_TRY(MakeStream(ctx_of('A'), &g.sA, pA));
      RFM_TRY(MakeStream(ctx_of('F'), &g.sF, pF));
      RFM_TRY(MakeStream(ctx_of('B'), &g.sB, pB));
      RFM_TRY(MakeStream(ctx_of('R'), &g.sR, pB));
      RFM_TRY(MakeStream(ctx_of('C'), &g.sC, pL));
      RFM_TRY(MakeStream(ctx_of('P'), &g.sP, pL));
      if (RFM_KNOB("RFM_DEBUG_SERIAL"))
      { // measurement aid: every stage on ONE stream, so per-kernel event times are isolated durations
        cudaStreamDestroy(g.sF); cudaStreamDestroy(g.sB); cudaStreamDestroy(g.sR); cudaStreamDestroy(g.sC); cudaStreamDestroy(g.sP);
        g.sF = g.sB = g.sR = g.sC = g.sP = g.sA;
      }
    }
    for (int b = 0; b < 2; ++b)
    {
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_front[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_demod[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_lanes[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_res[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_carry[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_pll[b], cudaEventDisableTiming));
      RFM_TRY(g.rlp_out[b].Alloc(S * d->nr_stride));
      RFM_TRY(g.lpS[b].Alloc(S * d->lp_stride));
      RFM_TRY(g.lpM[b].Alloc(S * d->lp_stride));
    }
    RFM_TRY(g.tail.Alloc(S * p.in_order));
    RFM_TRY(g.z[0].Alloc(S * d->z_stride));
    RFM_TRY(g.z[1].Alloc(S * d->z_stride));
    RFM_TRY(g.incr[0].Alloc(S * d->z_stride));
    RFM_TRY(g.incr[1].Alloc(S * d->z_stride));
    RFM_TRY(g.dm_start.Alloc(S * (size_t)demod_chunks(d->nb_max)));
    RFM_TRY(g.dm_end.Alloc(S * (size_t)demod_chunks(d->nb_max)));
    for (int b = 0; b < 3; ++b)
    {
      RFM_TRY(g.bbV[b].Alloc(S * d->a_stride));
      RFM_TRY(g.rawV[b].Alloc(S * d->a_stride));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_rest[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_rds[b], cudaEventDisableTiming));
      RFM_TRY(cudaEventCreateWithFlags(&g.ev_aud[b], cudaEventDisableTiming));
    }

    RFM_TRY(g.rlpV.Alloc(S * d->rlp_stride));
    RFM_TRY(g.rds_tails.Alloc(S * d->rds_tail_stride));
    RFM_TRY(g.mfV.Alloc(S * d->mf_stride));
    RFM_TRY(g.mf_out.Alloc(S * d->nr_stride));
    RFM_TRY(g.bits.Alloc(S * d->bits_cap));
    RFM_TRY(g.bit_count.Alloc(S));
    RFM_TRY(g.fS.Alloc(S * d->na_max));
    RFM_TRY(g.fM.Alloc(S * d->na_max));
    RFM_TRY(g.state.Alloc(S * SF_COUNT));
    RFM_TRY(ResetGroupState(d, g, true));
  }
  (void)esz_max;
  d->sync.resize(d->S);
  d->uecp.resize(d->S);
  d->host_bits.resize(d->S);
  RFM_TRY(cudaDeviceSynchronize());
#undef RFM_TRY
  *out = d;
  return RFM_OK;
}

void rfm_decoder_destroy(rfm_decoder* d) { FreeDecoder(d); }

int rfm_decoder_reset(rfm_decoder* d)
{
  if (!d)
    return Fail(RFM_ERR_INVALID, "null decoder");
  int rc = SyncAll(d);
  if (rc != RFM_OK)
    return rc;
  rc = DrainBits(d); // bits sliced before the reset belong to the old decoder state
  if (rc != RFM_OK)
    return rc;
  for (auto& g : d->groups)
    RFM_CUDA(ResetGroupState(d, g, false));
  d->rlp_g = 0; // InitLPFilter / InitConstFir reset m_State (FirFilter.cpp:145,319)
  d->mf_g = 0;
  for (auto& s : d->sync)
    s.Reset();
  // cFmDecoder::Reset -> cRDSRxSignalProcessor::Reset -> m_Decoder.Reset() (RDSProcess.cpp:92, RDSGroupDecoder.cpp:140-164):
  // PI / PS / TA_TP / MS / DI / PIN change detection, RadioText and ODA state start over.  Frames already handed out
  // (cRadioReceiver::AddUECPDataFrame has buffered them in the reference) stay in the pending byte stream.
  for (auto& u : d->uecp)
    u.Reset();
  return RFM_OK;
}

uint32_t rfm_decoder_max_audio_floats(const rfm_decoder* d, uint32_t n)
{
  if (!d)
    return 0;
  const unsigned nb = (n + d->plan.downsample - 1) / d->plan.downsample + 1;
  return 2 * ((unsigned)(nb / d->plan.a_ratio) + 4);
}

static int EnsureStaging(rfm_decoder* d, int fmt)
{
  const size_t esz = IqBytes(fmt);
  for (auto& g : d->groups)
  {
    const size_t need = (size_t)g.S * d->maxn * esz;
    if (g.in_stage.n < need)
    {
      g.in_stage.Free();
      RFM_CUDA(g.in_stage.Alloc(need));
    }
    if (g.audio_stage.n == 0)
      RFM_CUDA(g.audio_stage.Alloc((size_t)g.S * d->audio_cap));
  }
  return RFM_OK;
}

static bool KnownFormat(int fmt) { return fmt >= RFM_IQ_U8 && fmt <= RFM_IQ_CF32; }

// Host buffers of any format: staged into device memory (cudaMemcpyAsync) and decoded; `submit` only enqueues.
static int ProcessHost(rfm_decoder* d, int fmt, const void* iq, uint32_t n, float* audio, size_t audio_stride,
                       uint32_t* n_audio_floats, bool submit)
{
  if (!d || !iq || !audio)
    return Fail(RFM_ERR_INVALID, "null argument");
  if (!KnownFormat(fmt))
    return Fail(RFM_ERR_INVALID, "unknown IQ format");
  RFM_CUDA(cudaSetDevice(d->device));
  int rc = EnsureStaging(d, fmt);
  if (rc != RFM_OK)
    return rc;
  return ProcessDevice(d, iq, n, static_cast<IqFormat>(fmt), n, audio, audio_stride, n_audio_floats, nullptr, true, !submit);
}

int rfm_decoder_process_u8(rfm_decoder* d, const uint8_t* iq, uint32_t n, float* audio, size_t audio_stride,
                           uint32_t* n_audio_floats)
{
  return ProcessHost(d, RFM_IQ_U8, iq, n, audio, audio_stride, n_audio_floats, false);
}

int rfm_decoder_process_cf32(rfm_decoder* d, const float* iq, uint32_t n, float* audio, size_t audio_stride,
                             uint32_t* n_audio_floats)
{
  return ProcessHost(d, RFM_IQ_CF32, iq, n, audio, audio_stride, n_audio_floats, false);
}

int rfm_decoder_process_iq(rfm_decoder* d, int format, const void* iq, uint32_t n, float* audio, size_t audio_stride,
                           uint32_t* n_audio_floats)
{
  return ProcessHost(d, format, iq, n, audio, audio_stride, n_audio_floats, false);
}

int rfm_decoder_submit_u8(rfm_decoder* d, const uint8_t* iq, uint32_t n, float* audio, size_t audio_stride,
                          uint32_t* n_audio_floats)
{
  return ProcessHost(d, RFM_IQ_U8, iq, n, audio, audio_stride, n_audio_floats, true);
}

int rfm_decoder_submit_iq(rfm_decoder* d, int format, const void* iq, uint32_t n, float* audio, size_t audio_stride,
                          uint32_t* n_audio_floats)
{
  return ProcessHost(d, format, iq, n, audio, audio_stride, n_audio_floats, true);
}

int rfm_decoder_process_u8_device(rfm_decoder* d, const uint8_t* d_iq, size_t iq_stride, uint32_t n, float* d_audio,
                                  size_t audio_stride, uint32_t* n_audio_floats, void* cuda_stream)
{
  if (!d || !d_iq || !d_audio || iq_stride < n)
    return Fail(RFM_ERR_INVALID, "bad argument");
  return ProcessDevice(d, d_iq, iq_stride, kIqU8, n, d_audio, audio_stride, n_audio_floats,
                       static_cast<cudaStream_t>(cuda_stream), false);
}

int rfm_decoder_process_cf32_device(rfm_decoder* d, const float* d_iq, size_t iq_stride, uint32_t n, float* d_audio,
                                    size_t audio_stride, uint32_t* n_audio_floats, void* cuda_stream)
{
  if (!d || !d_iq || !d_audio || iq_stride < n)
    return Fail(RFM_ERR_INVALID, "bad argument");
  return ProcessDevice(d, d_iq, iq_stride, kIqCF32, n, d_audio, audio_stride, n_audio_floats,
                       static_cast<cudaStream_t>(cuda_stream), false);
}

int rfm_decoder_process_iq_device(rfm_decoder* d, int format, const void* d_iq, size_t iq_stride, uint32_t n,
                                  float* d_audio, size_t audio_stride, uint32_t* n_audio_floats, void* cuda_stream)
{
  if (!d || !d_iq || !d_audio || iq_stride < n)
    return Fail(RFM_ERR_INVALID, "bad argument");
  if (!KnownFormat(format))
    return Fail(RFM_ERR_INVALID, "unknown IQ format");
  // every sample is read with loads of its own size
  if (reinterpret_cast<uintptr_t>(d_iq) % IqBytes(format) != 0)
    return Fail(RFM_ERR_INVALID, "device IQ must be aligned to its sample size (2 / 2 / 4 / 8 bytes for u8 / s8 / s16 / cf32)");
  return ProcessDevice(d, d_iq, iq_stride, static_cast<IqFormat>(format), n, d_audio, audio_stride, n_audio_floats,
                       static_cast<cudaStream_t>(cuda_stream), false);
}

int rfm_decoder_wait(rfm_decoder* d, void* cuda_stream)
{
  if (!d)
    return Fail(RFM_ERR_INVALID, "null decoder");
  RFM_CUDA(cudaSetDevice(d->device));
  cudaStream_t user = static_cast<cudaStream_t>(cuda_stream);
  for (auto& g : d->groups)
  {
    cudaStream_t all[6];
    g.AllStreams(all);
    for (cudaStream_t st : all)
    {
      RFM_CUDA(cudaEventRecord(d->ev_join, st));
      RFM_CUDA(cudaStreamWaitEvent(user, d->ev_join, 0));
    }
  }
  return RFM_OK;
}

int rfm_decoder_demod_repairs(rfm_decoder* d, uint64_t* chunks)
{
  if (!d || !chunks)
    return Fail(RFM_ERR_INVALID, "bad argument");
  int rc = SyncAll(d);
  if (rc != RFM_OK)
    return rc;
  unsigned long long v = 0;
  RFM_CUDA(cudaMemcpy(&v, d->d_repairs.p, sizeof(v), cudaMemcpyDeviceToHost));
  *chunks = v;
  return RFM_OK;
}

int rfm_decoder_synchronize(rfm_decoder* d)
{
  if (!d)
    return Fail(RFM_ERR_INVALID, "null decoder");
  return SyncAll(d);
}

int rfm_decoder_rds_take_groups(rfm_decoder* d, uint32_t stream, uint16_t* groups, uint32_t max_groups,
                                uint32_t* n_groups)
{
  if (!d || stream >= d->S || !n_groups)
    return Fail(RFM_ERR_INVALID, "bad argument");
  int rc = SyncAll(d);
  if (rc == RFM_OK)
    rc = DrainBits(d);
  if (rc != RFM_OK)
    return rc;
  auto& g = d->sync[stream].Groups();
  const uint32_t n = std::min<uint32_t>((uint32_t)(g.size() / 4), max_groups);
  if (groups && n)
    memcpy(groups, g.data(), (size_t)n * 4 * sizeof(uint16_t));
  g.erase(g.begin(), g.begin() + (size_t)n * 4);
  *n_groups = n;
  return RFM_OK;
}

int rfm_decoder_rds_take_uecp(rfm_decoder* d, uint32_t stream, uint8_t* out, uint32_t cap, uint32_t* n_bytes)
{
  if (!d || stream >= d->S || !n_bytes)
    return Fail(RFM_ERR_INVALID, "bad argument");
  int rc = SyncAll(d);
  if (rc == RFM_OK)
    rc = DrainBits(d);
  if (rc != RFM_OK)
    return rc;
  auto& p = d->uecp[stream].Pending();
  const uint32_t n = (uint32_t)std::min<size_t>(p.size(), out ? cap : 0);
  if (n)
    memcpy(out, p.data(), n);
  p.erase(p.begin(), p.begin() + n);
  *n_bytes = n;
  return RFM_OK;
}

int rfm_decoder_rds_take_bits(rfm_decoder* d, uint32_t stream, uint8_t* bits, uint32_t max_bits, uint32_t* n_bits)
{
  if (!d || stream >= d->S || !n_bits)
    return Fail(RFM_ERR_INVALID, "bad argument");
  int rc = SyncAll(d);
  if (rc == RFM_OK)
    rc = DrainBits(d);
  if (rc != RFM_OK)
    return rc;
  auto& b = d->host_bits[stream];
  const uint32_t n = std::min<uint32_t>((uint32_t)b.size(), max_bits);
  if (bits && n)
    memcpy(bits, b.data(), n);
  b.erase(b.begin(), b.begin() + n);
  *n_bits = n;
  return RFM_OK;
}

int rfm_decoder_get_status(rfm_decoder* d, uint32_t stream, rfm_stream_status* out)
{
  if (!d || stream >= d->S || !out)
    return Fail(RFM_ERR_INVALID, "bad argument");
  unsigned ls = 0;
  Group* g = FindGroup(d, stream, &ls);
  RFM_CUDA(cudaSetDevice(d->device));
  {
    cudaStream_t all[6];
    g->AllStreams(all);
    for (cudaStream_t st : all)
      RFM_CUDA(cudaStreamSynchronize(st));
  }
  float v[SF_COUNT];
  RFM_CUDA(cudaMemcpy2D(v, sizeof(float), g->state.p + ls, (size_t)g->S * sizeof(float), sizeof(float), SF_COUNT,
                        cudaMemcpyDeviceToHost));
  int stereo;
  memcpy(&stereo, &v[SF_STEREO + ((d->block_index + 2) % 3u)], 4); // slot of the last block
  out->stereo_detected = stereo;
  out->interface_level = v[SF_IF_LEVEL];
  out->baseband_level = v[SF_BB_LEVEL];
  out->baseband_mean = v[SF_BB_MEAN];
  out->pilot_level = 2 * v[SF_PILOT_LEVEL];                                       // FmDecode.h:77
  const float tuned = -d->plan.tuning_shift * d->plan.fs_if / float(kTunerTable); // FmDecode.h:148
  out->tuning_offset = tuned + v[SF_BB_MEAN] * d->plan.freq_dev;
  return RFM_OK;
}

static int PlanConstants(const DecoderPlan& p, double* s, uint32_t max)
{
  if (!s || max < 51)
    return Fail(RFM_ERR_INVALID, "bad argument");
  int i = 0;
  s[i++] = p.fs_if; s[i++] = p.fs_bb; s[i++] = p.tuning_shift; s[i++] = p.demod_gain;
  s[i++] = p.nco_lo; s[i++] = p.nco_hi; s[i++] = p.pll_alpha; s[i++] = p.pll_beta; s[i++] = p.de_alpha;
  s[i++] = p.pilot.minfreq; s[i++] = p.pilot.maxfreq; s[i++] = p.pilot.b0; s[i++] = p.pilot.a1; s[i++] = p.pilot.a2;
  s[i++] = p.pilot.lb0; s[i++] = p.pilot.lb1; s[i++] = p.pilot.freq0; s[i++] = p.pilot.minsignal;
  s[i++] = p.pilot.lock_delay;
  s[i++] = p.in_order; s[i++] = p.downsample; s[i++] = p.a_order; s[i++] = p.a_ratio;
  s[i++] = p.rds_rate; s[i++] = p.rpll_lo; s[i++] = p.rpll_hi; s[i++] = p.rpll_alpha; s[i++] = p.rpll_beta;
  s[i++] = (double)p.mf_coef.size(); s[i++] = (double)p.rlp_coef.size();
  s[i++] = p.rds_osc.inc; s[i++] = p.rds_osc.cosv; s[i++] = p.rds_osc.sinv;
  s[i++] = p.rsync.A1; s[i++] = p.rsync.A2; s[i++] = p.rsync.B0; s[i++] = p.rsync.B1; s[i++] = p.rsync.B2;
  s[i++] = p.notch.A1; s[i++] = p.notch.A2; s[i++] = p.notch.B0; s[i++] = p.notch.B1; s[i++] = p.notch.B2;
  s[i++] = (double)p.lp_coef.size();
  s[i++] = (double)p.rds_stages.size();
  for (size_t k = 0; k < 6; ++k)
    s[i++] = k < p.rds_stages.size() ? p.rds_stages[k].len : 0;
  return i;
}

static int PlanTable(const DecoderPlan& p, int which, float* out, uint32_t max_floats, uint32_t* n)
{
  if (!n)
    return Fail(RFM_ERR_INVALID, "bad argument");
  const float* src = nullptr;
  size_t cnt = 0;
  switch (which)
  {
    case 0: src = p.tuner; cnt = 2 * kTunerTable; break;
    case 1: src = p.in_coeff.data(); cnt = p.in_coeff.size(); break;
    case 2: src = p.a_coeff.data(); cnt = p.a_coeff.size(); break;
    case 3: src = p.rlp_coef.data(); cnt = p.rlp_coef.size(); break;
    case 4: src = p.mf_coef.data(); cnt = p.mf_coef.size(); break;
    case 5: src = p.lp_coef.data(); cnt = p.lp_coef.size(); break;
    case 6: src = p.u8lut; cnt = 256; break;
    default: return Fail(RFM_ERR_INVALID, "unknown table");
  }
  cnt = std::min<size_t>(cnt, max_floats);
  if (out)
    memcpy(out, src, cnt * sizeof(float));
  *n = (uint32_t)cnt;
  return RFM_OK;
}

static int PlanFromConfig(const rfm_config* cfg, DecoderPlan* plan)
{
  if (!cfg || cfg->downsample == 0 || cfg->sample_rate_if <= 0 || cfg->sample_rate_pcm <= 0)
    return Fail(RFM_ERR_INVALID, "invalid configuration");
  *plan = PlanDecoder(cfg->sample_rate_if, cfg->tuning_offset, cfg->sample_rate_pcm, cfg->bandwidth_pcm,
                      cfg->downsample, cfg->us_deemphasis != 0);
  return RFM_OK;
}

int rfm_plan_constants(const rfm_config* cfg, double* s, uint32_t max)
{
  DecoderPlan plan;
  const int rc = PlanFromConfig(cfg, &plan);
  return rc != RFM_OK ? rc : PlanConstants(plan, s, max);
}

int rfm_plan_table(const rfm_config* cfg, int which, float* out, uint32_t max_floats, uint32_t* n)
{
  DecoderPlan plan;
  const int rc = PlanFromConfig(cfg, &plan);
  return rc != RFM_OK ? rc : PlanTable(plan, which, out, max_floats, n);
}

int rfm_decoder_constants(const rfm_decoder* d, double* s, uint32_t max)
{
  if (!d)
    return Fail(RFM_ERR_INVALID, "bad argument");
  return PlanConstants(d->plan, s, max);
}

int rfm_decoder_table(const rfm_decoder* d, int which, float* out, uint32_t max_floats, uint32_t* n)
{
  if (!d)
    return Fail(RFM_ERR_INVALID, "bad argument");
  return PlanTable(d->plan, which, out, max_floats, n);
}

/* A stream on the FIR side of the decoder's SM partition (an ordinary non-blocking stream when the decoder has none),
 * for the caller's own kernels that produce the decoder's input (e.g. rfm_downconvert in front of
 * rfm_decoder_process_cf32_device): what runs there never shares an SM with the lanes kernel.  Owned by the decoder. */
int rfm_decoder_companion_stream(rfm_decoder* d, void** stream)
{
  if (!d || !stream)
    return Fail(RFM_ERR_INVALID, "bad argument");
  if (!d->s_companion)
  {
    RFM_CUDA(cudaSetDevice(d->device));
    int prio_lo = 0, prio_hi = 0;
    RFM_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    RFM_CUDA(MakeStream(d->part.rest, &d->s_companion, prio_lo));
  }
  *stream = d->s_companion;
  return RFM_OK;
}

int rfm_decoder_set_profiling(rfm_decoder* d, int on)
{
  if (!d)
    return Fail(RFM_ERR_INVALID, "null decoder");
  int rc = SyncAll(d);
  if (rc != RFM_OK)
    return rc;
  for (auto& g : d->groups)
    ProfCollect(d, g.prof);
  ProfCollect(d, d->main_prof);
  memset(d->prof_ms, 0, sizeof(d->prof_ms));
  memset(d->prof_count, 0, sizeof(d->prof_count));
  d->profiling = on != 0;
  if (on)
  {
    if (!d->ev_base)
      cudaEventCreate(&d->ev_base);
    cudaEventRecord(d->ev_base, d->s_osc);
  }
  return RFM_OK;
}

int rfm_decoder_profile_read(rfm_decoder* d, uint32_t index, char* name, uint32_t name_cap, double* total_ms,
                             uint64_t* launches)
{
  if (!d || !name || name_cap == 0 || !total_ms || !launches)
    return Fail(RFM_ERR_INVALID, "bad argument");
  if (index == 0)
  {
    int rc = SyncAll(d);
    if (rc != RFM_OK)
      return rc;
    for (auto& g : d->groups)
      ProfCollect(d, g.prof);
    ProfCollect(d, d->main_prof);
  }
  if (index >= (uint32_t)kMaxProfKinds || !d->prof_names[index])
    return 1; // end of list
  snprintf(name, name_cap, "%s", d->prof_names[index]);
  *total_ms = d->prof_ms[index];
  *launches = d->prof_count[index];
  return RFM_OK;
}

int rfm_decoder_tap(rfm_decoder* d, const char* name, uint32_t stream, float* out, uint32_t max_floats,
                    uint32_t* n_floats)
{
  if (!d || !name || stream >= d->S || !out || !n_floats)
    return Fail(RFM_ERR_INVALID, "bad argument");
  int rc = SyncAll(d);
  if (rc != RFM_OK)
    return rc;
  unsigned ls = 0;
  Group* g = FindGroup(d, stream, &ls);
  const DecoderPlan& p = d->plan;
  const std::string nm(name);
  const unsigned lastpar = (unsigned)((d->block_index + 1) & 1u);
  const unsigned lastpar3 = (unsigned)((d->block_index + 2) % 3u);
  const void* src = nullptr;
  size_t cnt = 0; // floats
  if (nm == "demod_in") { src = g->z[lastpar].p + (size_t)ls * d->z_stride; cnt = 2 * (size_t)d->last_nb; }
  else if (nm == "baseband") { src = g->bbV[lastpar3].p + (size_t)ls * d->a_stride + p.a_order; cnt = d->last_nb; }
  else if (nm == "rawstereo") { src = g->rawV[lastpar3].p + (size_t)ls * d->a_stride + p.a_order; cnt = d->last_nb; }
  else if (nm == "mono_rs") { src = g->lpM[(d->block_index + 1) & 1u].p + (size_t)ls * d->lp_stride + p.lp_coef.size() - 1; cnt = d->last_na; }
  else if (nm == "stereo_rs") { src = g->lpS[(d->block_index + 1) & 1u].p + (size_t)ls * d->lp_stride + p.lp_coef.size() - 1; cnt = d->last_na; }
  else if (nm == "lp_stereo") { src = g->fS.p + (size_t)ls * d->na_max; cnt = d->last_na; }
  else if (nm == "lp_mono") { src = g->fM.p + (size_t)ls * d->na_max; cnt = d->last_na; }
  else if (nm == "rds_dec") { src = g->rlpV.p + (size_t)ls * d->rlp_stride + p.rlp_coef.size() - 1; cnt = 2 * (size_t)d->last_nr; }
  else if (nm == "rds_lp") { src = g->rlp_out[(d->block_index + 1) & 1u].p + (size_t)ls * d->nr_stride; cnt = 2 * (size_t)d->last_nr; }
  else if (nm == "rds_pll") { src = g->mfV.p + (size_t)ls * d->mf_stride + p.mf_coef.size() - 1; cnt = d->last_nr; }
  else if (nm == "rds_mf") { src = g->mf_out.p + (size_t)ls * d->nr_stride; cnt = d->last_nr; }
  else
    return Fail(RFM_ERR_INVALID, "unknown tap name");
  if (cnt > max_floats)
    return Fail(RFM_ERR_OVERFLOW, "tap buffer too small");
  RFM_CUDA(cudaMemcpy(out, src, cnt * sizeof(float), cudaMemcpyDeviceToHost));
  *n_floats = (uint32_t)cnt;
  return RFM_OK;
}

// ---- host-only RDS block sync ---------------------------------------------------------------------------
struct rfm_rdssync
{
  RdsBlockSync s;
};

int rfm_rdssync_create(rfm_rdssync** out)
{
  if (!out)
    return Fail(RFM_ERR_INVALID, "null argument");
  *out = new rfm_rdssync;
  return RFM_OK;
}
void rfm_rdssync_destroy(rfm_rdssync* s) { delete s; }
void rfm_rdssync_reset(rfm_rdssync* s)
{
  if (s)
    s->s.Reset();
}
int rfm_rdssync_push_bits(rfm_rdssync* s, const uint8_t* bits, uint32_t n)
{
  if (!s || (!bits && n))
    return Fail(RFM_ERR_INVALID, "bad argument");
  for (uint32_t i = 0; i < n; ++i)
    s->s.PushBit(bits[i] & 1);
  return RFM_OK;
}
int rfm_rdssync_take_groups(rfm_rdssync* s, uint16_t* groups, uint32_t max_groups, uint32_t* n_groups)
{
  if (!s || !n_groups)
    return Fail(RFM_ERR_INVALID, "bad argument");
  auto& g = s->s.Groups();
  const uint32_t n = std::min<uint32_t>((uint32_t)(g.size() / 4), max_groups);
  if (groups && n)
    memcpy(groups, g.data(), (size_t)n * 4 * sizeof(uint16_t));
  g.erase(g.begin(), g.begin() + (size_t)n * 4);
  *n_groups = n;
  return RFM_OK;
}
uint32_t rfm_rds_check_block(uint32_t word26, uint32_t offset_syndrome, int use_fec, uint32_t* corrected)
{
  uint32_t w = word26;
  const uint32_t syn = RdsCheckBlock(&w, offset_syndrome, use_fec != 0);
  if (corrected)
    *corrected = w;
  return syn;
}

} // extern "C"
