// rfm_kernels.cuh -- launch interface of the sm_100a kernels (rfm_kernels.cu).
//
// Data layout (all batched [stream][time], one row per IQ stream, everything resident in HBM):
//   * "V buffers": a stage's input row is  [ H history samples | n new samples ]  so that a FIR tile
//     can read across the block boundary without branching; the producer writes at offset H and
//     k_tails moves the last H samples to the front after the consumer has run
//     (the reference's m_state / m_pHBFirBuf / m_cZBuf carry, DownConvert.cpp:135-153,544-547).
//   * per-stream scalar state (PLL registers, IIR delays, meters) lives in SoA float arrays.
//   * state that depends only on the number of samples processed (fine-tuner index, decimator
//     phase, fractional resampler position, FIR rotation, NCO-oscillator phasor) is identical for
//     all streams of a decoder and is tracked once (host scalars / one device table).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "rfm_math.cuh"
#include "rfm_steps.cuh"

namespace rfm
{

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device, per-function setting: remember the largest value set
// for every (device, function) pair, so that decoders on several devices of one process (and several host threads)
// all get it.  Cheap enough for every launch (one cudaGetDevice + a map lookup under a mutex).
void EnsureDynSmemImpl(const void* func, size_t smem);
template <typename F>
inline void EnsureDynSmem(F* func, size_t smem)
{
  EnsureDynSmemImpl(reinterpret_cast<const void*>(func), smem);
}


// Measurement knobs (RFM_DEBUG_* / RFM_LANES_* / ... environment variables) exist only in the experiments build
// (RFM_EXPERIMENTS=1 sh build.sh -> libradiofm_b200_exp.so).  The product library reads no environment variable:
// RFM_KNOB(name) is a null constant there and every branch that depends on one is compiled out.
#ifdef RFM_EXPERIMENTS
#define RFM_KNOB(name) getenv(name)
#else
#define RFM_KNOB(name) (static_cast<const char*>(nullptr))
#endif
inline int KnobInt(const char* v, int dflt) { return v ? atoi(v) : dflt; }

constexpr unsigned kMaxFirTapsDev = 80; // >= cFirFilter MAX_NUMCOEF (75)

// ---- per-stream scalar state, SoA: state[field * S + stream] --------------------------------------
enum StateField
{
  SF_DEMOD_PHASE = 0,
  SF_DEMOD_INCR,
  SF_DEMOD_DC,
  SF_IF_LEVEL,
  SF_BB_MEAN,
  SF_BB_LEVEL,
  SF_PILOT_PHASE,
  SF_PILOT_FREQ,
  SF_PILOT_I1,
  SF_PILOT_I2,
  SF_PILOT_Q1,
  SF_PILOT_Q2,
  SF_PILOT_X1,
  SF_PILOT_LEVEL,
  SF_PILOT_LOCKCNT, // int bits
  SF_STEREO,        // int bits: m_StereoDetected of the last block (even blocks)
  SF_STEREO1,       // ... three slots by block index mod 3 (the lanes of blocks k+1, k+2 overlap the audio tail of block k)
  SF_STEREO2,
  SF_DE_RE,
  SF_DE_IM,
  SF_NOTCH_W1A,
  SF_NOTCH_W2A,
  SF_NOTCH_W1B,
  SF_NOTCH_W2B,
  SF_RPLL_PHASE,
  SF_RPLL_FREQ,
  SF_RSYNC_W1,
  SF_RSYNC_W2,
  SF_RS_LASTSYNC,
  SF_RS_LASTSLOPE,
  SF_RS_LASTDATA,
  SF_RS_LASTBIT, // int bits
  SF_COUNT
};

// ---- front end: (u8 | s8 | s16 | cf32) -> fine tuner -> Lanczos FIR / ds ---------------------------------
struct FrontParams
{
  const void* in;          // [S][in_stride] samples of the IQ format (rfm_dsp.cuh IqFormat)
  size_t in_stride;        // samples per row
  unsigned n;              // new samples per stream
  unsigned S;
  unsigned order, ds;
  unsigned p0;             // m_pos_int: position of the first output inside this block
  unsigned nout;           // outputs per stream
  unsigned idx0;           // fine-tuner table index of sample 0
  const float* lut;        // [256]
  const float* tuner;      // [64][2]
  const float* coeff;      // [order + 2] (device)
  const float* coeff_host; // the same table on the host (kernel-parameter constant bank of the tiled kernel)
  cf32* tail;              // [S][order] tuned history (m_stateComplex)
  cf32* z;                 // [S][z_stride] FIR output
  size_t z_stride;
  unsigned sm_count = 0;   // SMs of the launching stream's partition (0: the whole device); sizes persistent grids
  bool fused = false;      // tolerance mode (rfm_config::fir_fused): FFMA in the FIR, not bit-exact
};
enum IqFormat : int; // rfm_dsp.cuh (an enum, so that no bool or stray integer converts to a format)
void launch_front(const FrontParams& p, IqFormat fmt, cudaStream_t st);
void launch_front_tail(const FrontParams& p, IqFormat fmt, cudaStream_t st);

// ---- baseband lanes: IF meter, FM-demod PLL, DC tracker, BB meters, pilot PLL, 38 kHz demux multiply --
void launch_if_level(const FrontParams& p, float* state, IqFormat fmt, cudaStream_t st);

// ---- FM-demodulator PLL: speculative chunk-parallel pass + exactness check / sequential repair --------------------
struct DemodSpecParams
{
  const cf32* z;           // [S][z_stride] decimated IQ
  size_t z_stride;
  unsigned nb, S;
  unsigned warm;           // speculative warm-up samples (multiple of 32, <= 192)
  float* state;            // [SF_COUNT][S]: SF_DEMOD_PHASE / SF_DEMOD_INCR carried
  DemodConst demod;
  float* incr;             // [S][w_stride] NCO increment after every sample
  size_t w_stride;
  float2* st_start;        // [chunks][S] state a chunk assumed at its first sample
  float2* st_end;          // [chunks][S] state after its last sample
  unsigned long long* repairs; // telemetry: chunks that had to be recomputed sequentially (may be null)
};
void launch_demod_spec(const DemodSpecParams& p, cudaStream_t st);
void launch_demod_fix(const DemodSpecParams& p, cudaStream_t st);
unsigned demod_chunks(unsigned nb);

struct LanesParams
{
  const float* incr;       // [S][w_stride] from the demodulator
  size_t w_stride;
  unsigned nb;             // baseband samples per stream
  unsigned S;
  float* state;            // [SF_COUNT][S]
  DemodConst demod;
  PilotConstDev pilot;
  float* bbV;              // [S][a_stride]: history a_hist, then nb new baseband samples
  float* rawV;             // same layout, pilot-demodulated L-R
  size_t a_stride;
  unsigned a_hist;
  unsigned parity;         // selects SF_STEREO / SF_STEREO1
  bool packed;             // the lanes stream lives in an SM partition: use the immediate-barrier kernel (12 CTAs per SM)
  unsigned role_swap;      // set by launch_bb_lanes: odd CTAs run the pilot PLL on warp 0 (RFM_LANES_SWAP, experiment)
};
void launch_bb_lanes(const LanesParams& p, cudaStream_t st);

// ---- audio: fractional Lanczos resampler (mono + stereo share the interpolated taps) -------------------
struct ResampleParams
{
  const float* bbV;
  const float* rawV;
  size_t a_stride;
  unsigned order;          // V history length == order
  unsigned nb, S, na;
  float pos_frac, pstep;
  const float* coeff;      // [order + 2]
  float* lpS;              // [S][lp_stride]: history (lp_taps - 1), then na new samples (stereo diff)
  float* lpM;              // same, mono
  size_t lp_stride;
  unsigned lp_hist;
  // tiled form: per-block tap table shared by all streams (launch_res_taps)
  const float* kk;         // [groups][lp][4]
  const int* meta;         // [groups][2]: first V index, length
  unsigned lp;             // time steps reserved per group (>= order + 1 + 3 * ceil(ratio) + 1)
  bool fused = false;      // tolerance mode
};
void launch_resample(const ResampleParams& p, cudaStream_t st);
void launch_resample_tiled(const ResampleParams& p, cudaStream_t st);

struct ResTapsParams
{
  float pos_frac, pstep;
  unsigned na, order, lp;
  const float* coeff;      // [order + 2]
  float* kk;
  int* meta;
};
void launch_res_taps(const ResTapsParams& p, cudaStream_t st);

// ---- cFirFilter with rotating summation start (real pair / complex / real) ------------------------------
struct RotFirParams
{
  const float* inA;        // V rows: history (taps - 1) then n
  const float* inB;        // second channel or nullptr
  size_t in_stride;        // in elements (float, or cf32 when cplx)
  float* outA;
  float* outB;
  size_t out_stride;
  unsigned out_off;        // element offset inside the output row (history of the consumer)
  unsigned n, S, taps;
  unsigned g0;             // samples filtered since the last (re)initialisation, mod taps
  const float* coef;       // [taps]
  int cplx;                // 1: rows are cf32, same taps for re and im
  bool fused = false;      // tolerance mode
};
void launch_rotfir(const RotFirParams& p, cudaStream_t st);

// ---- audio tail lanes: deemphasis, 19 kHz notch, L/R matrix -------------------------------------------
struct AudioTailParams
{
  const float* inS;
  const float* inM;
  size_t in_stride;
  unsigned na, S;
  float* state;
  float de_alpha;
  BiquadDev notch;
  float* audio;            // [S][audio_stride] interleaved L,R
  size_t audio_stride;
  unsigned parity;         // selects SF_STEREO / SF_STEREO1
};
void launch_audio_tail(const AudioTailParams& p, cudaStream_t st);

// ---- RDS: NCO oscillator table, half-band chain, PLL, slicer ------------------------------------------
struct OscParams
{
  cf32* oscV;              // [osc_hist + nb]
  unsigned osc_hist, nb;
  float* osc1;             // [2] carried phasor m_Osc1
  float cosv, sinv;
};
void launch_osc(const OscParams& p, cudaStream_t st);

// fused RDS front: mix + decimate-by-2 chain + RDS low-pass, histories carried in a per-stream tail row
constexpr unsigned kRfMaxStages = 6;
struct RdsFrontStage
{
  int kind;                // 0 generic half-band, 1 fixed 11-tap, 2 CIC3
  unsigned len, hist;
  const float* h;          // device taps (nullptr for CIC3)
  const float* h_host;     // the same taps on the host (constant-bank form of the register-tiled kernel), may be nullptr
};
struct RdsFrontParams
{
  const float* bbV;        // [S][a_stride], new samples at a_hist
  size_t a_stride;
  unsigned a_hist;
  const cf32* osc;         // NCO phasors of this block (first new sample)
  unsigned nb, S, nst;
  RdsFrontStage st[kRfMaxStages];
  const float* lp_coef;    // RDS LP taps (device)
  unsigned lp_n, g0;       // g0: samples filtered since the LP was (re)initialised, mod lp_n
  cf32* tails;             // [S][tail_stride]: per-stage histories, then the LP delay line
  size_t tail_stride;
  unsigned tail_off[kRfMaxStages + 1];
  cf32* out;               // [S][out_stride] LP output
  cf32* dec_out;           // [S][out_stride] decimator output (optional, for the stage taps)
  size_t out_stride;
  unsigned short_mask;     // bit k: stage k gets fewer samples than its FIR is long this block -> passes the first half through
  cf32* lp_v;              // when set: the last stage's outputs go to this V buffer ([lp_n - 1 history | n] rows) and the LP
  size_t lp_v_stride;      // is NOT applied here (the caller runs launch_rotfir on it); `out` / the LP tail are unused
};
void launch_rds_front(const RdsFrontParams& p, cudaStream_t st);

struct RdsPllParams
{
  const cf32* in;          // [S][in_stride]
  size_t in_stride;
  unsigned nr, S;
  float* state;
  float lo, hi, alpha, beta;
  float* out;              // matched-filter V buffer
  size_t out_stride;
  unsigned out_off;
};
void launch_rds_pll(const RdsPllParams& p, cudaStream_t st);

struct RdsSliceParams
{
  const float* in;         // matched filter output [S][in_stride]
  size_t in_stride;
  unsigned nr, S;
  float* state;
  BiquadDev sync;
  uint8_t* bits;           // [S][bits_cap]
  unsigned bits_cap;
  unsigned* bit_count;     // [S] running count (appended across blocks until drained)
};
void launch_rds_slice(const RdsSliceParams& p, cudaStream_t st);

// ---- history carry for V buffers -------------------------------------------------------------------------
struct TailDesc
{
  void* base;              // source rows: [hist | n]
  void* dst;               // destination rows (== base for an in-place carry)
  size_t stride_bytes;     // row stride (same for both)
  unsigned hist;           // elements of history
  unsigned n;              // new elements this block
  unsigned elem;           // element size in bytes (4 or 8)
  unsigned rows;           // S, or 1 for shared tables
};
constexpr int kMaxTailDesc = 12;
struct TailParams
{
  TailDesc d[kMaxTailDesc];
  int count;
};
void launch_tails(const TailParams& p, unsigned S, cudaStream_t st);

} // namespace rfm
