/* radiofm_b200.h -- C ABI of the B200-native IQ -> audio (+RDS) chain.
 *
 * Drop-in boundary for the DSP path of AlwinEsch/pvr.rtl.radiofm (SURVEY.md section 8b).  The reference
 * has no FFI seam: its DSP is a set of C++ classes linked into the add-on.  The replacement keeps
 * those class signatures in host C++ (pvr.rtl.radiofm_b200/host/<same-named>.h) as one-line forwards
 * onto the entry points below; each entry point cites the reference interface it replaces
 * (paths relative to the reference's src/).  Plain pointers and sizes only.
 *
 * Conventions
 *   - IQ in : interleaved I,Q, little-endian, in one of the rfm_iq_format formats below.  The _u8 / _cf32 entry points
 *             are the reference's two (u8 offset-binary from the RTL-SDR, 127.5 == 0; float32 complex); the _iq entry
 *             points take the format as an argument.
 *   - audio : interleaved float32 L,R at sample_rate_pcm.
 *   - Batched: a decoder handle owns n_streams independent streams that are always processed with
 *     the same block length (row-major [stream][sample]).  n_streams == 1 reproduces one cFmDecoder.
 *   - Every function returns RFM_OK (0) or a negative rfm_status; CUDA failures are RFM_ERR_CUDA and
 *     rfm_last_error() gives the text.  There is NO CPU fallback: without a usable sm_100 device the
 *     create calls fail.
 *   - "_device" variants take device pointers and a cudaStream_t (as void*) and only enqueue work.
 */
#ifndef RADIOFM_B200_H
#define RADIOFM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RFM_API __attribute__((visibility("default")))

typedef enum rfm_status
{
  RFM_OK = 0,
  RFM_ERR_INVALID = -1,     /* bad argument */
  RFM_ERR_CUDA = -2,        /* CUDA runtime error, see rfm_last_error() */
  RFM_ERR_UNSUPPORTED = -3, /* block shape the batched path does not implement (see DESIGN.md) */
  RFM_ERR_NO_DEVICE = -4,   /* no sm_100 device / extension unusable */
  RFM_ERR_OVERFLOW = -5     /* caller buffer too small */
} rfm_status;

/* IQ sample formats (interleaved I,Q, little-endian):
 *   RFM_IQ_U8    RTL-SDR offset binary, float(u / 127.5 - 1) (RTL_SDR_Source.cpp:207-211)
 *   RFM_IQ_S8    cs8 (HackRF), (float)v * 2^-7
 *   RFM_IQ_S16   cs16 (USRP, bladeRF, LimeSDR, Airspy, SDRplay: the SoapySDR / UHD host format), (float)v * 2^-15
 *   RFM_IQ_CF32  float32 complex, taken as is
 * The s8 / s16 conversions are exact in float32: an s8 / s16 input gives bit for bit what the cf32 path gives for the
 * converted samples.  Full scale is the container's: a stream that uses fewer bits (bladeRF SC16_Q11: 12 bits in 16)
 * reads 2^(16-12) = 24 dB low; levels and the scan's dBFS values are relative to the container.
 * Value domain: every code of every format and every finite float (zeros of either sign, subnormals, magnitudes up to
 * FLT_MAX) gives the reference's outputs bit for bit.  Where the reference's arithmetic itself makes a NaN (a NaN or
 * Inf sample, or an overflow inside the chain), the outputs are NaN-equivalent to it: NaN at the same places, every
 * other value bit-equal (the NaN bit patterns are the device's).  The calls return RFM_OK; a NaN stays in its stream
 * as in the reference (rfm_decoder_reset, like cFmDecoder::Reset, leaves the filters' delay lines and the de-emphasis
 * state as they are: only a new decoder starts clean), and the band scan refuses a non-finite spectrum
 * (rfm_scan_run).  rfm_iq_estimate on a non-finite cf32 capture returns a non-finite dc, a = 1, b = 0 and
 * imbalance_valid = 0. */
typedef enum rfm_iq_format { RFM_IQ_U8 = 0, RFM_IQ_S8 = 1, RFM_IQ_S16 = 2, RFM_IQ_CF32 = 3 } rfm_iq_format;
/* bytes per complex sample: 2, 2, 4, 8; 0 for an unknown format */
RFM_API uint32_t rfm_iq_format_bytes(int format);

/* IQ correction: the DC offset and the IQ gain / phase imbalance of a zero-IF receiver (HackRF, bladeRF, E4000 tuners),
 * frequency-flat, one set of coefficients per capture.  Off by default everywhere.
 *   Application  right after the format conversion, in float32, each step rounded on its own (no contraction):
 *                r = I - dc_i, q = Q - dc_q, y = r + j (a q + b r).  Before the pre-mix table and the NCO.
 *   Estimate     (rfm_iq_estimate) means m_I, m_Q and centred moments v_I, v_Q, c = E[I0 Q0] of the capture;
 *                dc = (m_I, m_Q), a = sqrt(v_I / (v_Q - c^2 / v_I)), b = -a c / v_I (Gram-Schmidt: y is proper, its
 *                real and imaginary parts uncorrelated with equal power).  Every value is computed in double and rounded
 *                to float once.  v_I = 0 or v_I v_Q - c^2 <= 0 (or a non-finite result): a = 1, b = 0,
 *                imbalance_valid = 0.  u8 / s8 / s16: 64-bit integer sums of codes, squares and cross products, centred
 *                moments n S_xx - S_x S_y in 128-bit integers, then scaled -- bit-identical on any device and work
 *                split; n <= 2^32.  cf32: double sums in an order that depends on n only.  oracle/iqcorr.py restates
 *                both.
 * Not covered: the decoder's own front end (rfm_decoder_*), frequency-dependent imbalance, tracking over time. */
typedef struct rfm_iq_correction
{
  float dc_i, dc_q;         /* subtracted after the format conversion */
  float a, b;               /* y = (I - dc_i) + j (a (Q - dc_q) + b (I - dc_i)) */
  int32_t imbalance_valid;  /* 0: a = 1, b = 0 were forced (degenerate statistics) */
} rfm_iq_correction;
/* One pass over n samples of `format`, in host memory (copied to `device`) or device memory (complete before the call,
 * aligned to the sample size).  Blocking.  RFM_ERR_INVALID for an unknown format, a misaligned device pointer, n = 0 or
 * n > 2^32, with the reason in rfm_last_error().  device: -1 = current. */
RFM_API int rfm_iq_estimate(int format, const void* iq, uint64_t n, int iq_on_device, int device, rfm_iq_correction* out);

RFM_API const char* rfm_last_error(void);
RFM_API const char* rfm_version(void);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
RFM_API uint64_t rfm_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * cFmDecoder (FmDecode.h:99-165, FmDecode.cpp:237-539), batched
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_decoder rfm_decoder;

typedef struct rfm_config
{
  double sample_rate_if;   /* cFmDecoder ctor arg, FmDecode.h:110-116 */
  double tuning_offset;
  double sample_rate_pcm;
  double bandwidth_pcm;    /* DEFAULT_BANDWIDTH_PCM 15000 */
  uint32_t downsample;     /* >= 1 */
  int32_t us_deemphasis;   /* USver: 75 us instead of 50 us */
  uint32_t n_streams;      /* >= 1 */
  uint32_t max_block_len;  /* largest n per call; the reference's limit is 65536 (FmDecode.cpp:277) */
  int32_t device;          /* CUDA device ordinal, -1 = current */
  uint32_t n_groups;       /* internal stream groups pipelined on separate CUDA streams, 0 = one group.  Device-pointer
                            * callers want 1 (every group pays the lanes kernel's ~1 ms latency chain); host-buffer
                            * callers of a wide batch want ~4, so that the H2D copy of one group overlaps the kernels of
                            * the others (4096 streams: blocking call 12.0 ms with 4, 13.9 with 1, 14.3 with 8) */
  uint32_t lanes_sms;      /* SM partition: the one-lane-per-stream recurrences (pilot PLL / DC tracker) run in a
                            * green context of this many SMs (multiple of 8, >= 8), every FIR kernel in the rest, so
                            * neither waits for the other's issue slots.  0 = automatic (24 SMs when n_streams >= 2048
                            * on a device of >= 100 SMs, none otherwise), 1 = never.  Placement only: results are
                            * identical.  Ignored (rfm_last_error says why, creation still succeeds) when the driver
                            * has no green contexts. */
  uint32_t fir_fused;      /* 0 (default): every multiply and add of the FIRs is rounded on its own, in the reference's
                            * order -- results bit-identical to the reference.  1: TOLERANCE MODE -- the front-end FIR,
                            * the fractional resamplers and the rotating FIRs use fused multiply-adds (half the
                            * instructions).  Audio then differs from the reference by ~1e-4 of full scale (typical
                            * streams stay inside BASELINE.json's 1e-4; the worst of 4096 reached 1.75e-4: DESIGN.md
                            * section 11), RDS bits normally still agree; not covered by the bit-exact parity tests.
                            * After a NaN or Inf sample the resamplers may also place NaN up to 3 outputs early. */
} rfm_config;

RFM_API void rfm_config_default(rfm_config* cfg);

/* new cFmDecoder(proc, sample_rate_if, tuning_offset, sample_rate_pcm, bandwidth_pcm, downsample, USver)
 * -- RadioReceiver.cpp:296-300 */
RFM_API int rfm_decoder_create(const rfm_config* cfg, rfm_decoder** out);
/* delete m_FMDecoder -- RadioReceiver.cpp:371-374 */
RFM_API void rfm_decoder_destroy(rfm_decoder* d);
/* cFmDecoder::Reset -- FmDecode.cpp:326-338 (clears meters, demod PLL and the RDS receiver only) */
RFM_API int rfm_decoder_reset(rfm_decoder* d);

/* Upper bound of audio floats per stream for a block of n samples (caller allocates; the reference's
 * caller allocates 2*n, RadioReceiver.cpp:519-520). */
RFM_API uint32_t rfm_decoder_max_audio_floats(const rfm_decoder* d, uint32_t n);

/* cRtlSdrSource::ReadAsyncCB conversion (RTL_SDR_Source.cpp:196-213) fused with
 * cFmDecoder::ProcessStream (FmDecode.cpp:417-502).  Host buffers:
 *   iq    [n_streams][n][2] u8
 *   audio [n_streams][audio_stride] float, audio_stride >= *n_audio_floats
 * *n_audio_floats = floats written per stream (2 x frames; identical for all streams). */
RFM_API int rfm_decoder_process_u8(rfm_decoder* d, const uint8_t* iq, uint32_t n, float* audio,
                                   size_t audio_stride, uint32_t* n_audio_floats);
/* unsigned ProcessStream(const ComplexType* samples_in, unsigned samples, float* audio)
 * -- FmDecode.h:135; iq is [n_streams][n] complex float. */
RFM_API int rfm_decoder_process_cf32(rfm_decoder* d, const float* iq, uint32_t n, float* audio,
                                     size_t audio_stride, uint32_t* n_audio_floats);

/* Asynchronous form of rfm_decoder_process_u8 for batch serving: the block is only enqueued (H2D copy, kernels, D2H
 * copy), so that the copy of block k+1 overlaps the kernels of block k.  iq should be pinned host memory; iq and
 * audio must stay valid / untouched until rfm_decoder_synchronize() returns. */
RFM_API int rfm_decoder_submit_u8(rfm_decoder* d, const uint8_t* iq, uint32_t n, float* audio, size_t audio_stride,
                                  uint32_t* n_audio_floats);

/* Same with device-resident buffers.  The call only ENQUEUES the block: it is ordered after everything already
 * submitted to `cuda_stream` (cudaStream_t), runs on the decoder's own streams (so that consecutive blocks
 * pipeline: the PLL lanes of block k+1 overlap the FIR stages of block k) and returns at once.  The caller
 * orders its own work after the results with rfm_decoder_wait(), or blocks with rfm_decoder_synchronize();
 * d_iq must stay untouched until then.  iq_stride is in samples per stream row; d_audio rows must be 8-byte
 * aligned (even audio_stride). */
RFM_API int rfm_decoder_process_u8_device(rfm_decoder* d, const uint8_t* d_iq, size_t iq_stride, uint32_t n,
                                          float* d_audio, size_t audio_stride, uint32_t* n_audio_floats,
                                          void* cuda_stream);
RFM_API int rfm_decoder_process_cf32_device(rfm_decoder* d, const float* d_iq, size_t iq_stride, uint32_t n,
                                            float* d_audio, size_t audio_stride, uint32_t* n_audio_floats,
                                            void* cuda_stream);
/* The three calls above for any rfm_iq_format: iq is [n_streams][n] samples of `format` (iq_stride in samples).  An
 * unknown format returns RFM_ERR_INVALID; so does a device pointer that is not aligned to the sample size
 * (rfm_iq_format_bytes). */
RFM_API int rfm_decoder_process_iq(rfm_decoder* d, int format, const void* iq, uint32_t n, float* audio,
                                   size_t audio_stride, uint32_t* n_audio_floats);
RFM_API int rfm_decoder_submit_iq(rfm_decoder* d, int format, const void* iq, uint32_t n, float* audio,
                                  size_t audio_stride, uint32_t* n_audio_floats);
RFM_API int rfm_decoder_process_iq_device(rfm_decoder* d, int format, const void* d_iq, size_t iq_stride, uint32_t n,
                                          float* d_audio, size_t audio_stride, uint32_t* n_audio_floats,
                                          void* cuda_stream);

/* Make `cuda_stream` wait for every block enqueued so far (no host blocking) / block the host until done. */
RFM_API int rfm_decoder_wait(rfm_decoder* d, void* cuda_stream);
RFM_API int rfm_decoder_synchronize(rfm_decoder* d);

/* RDS output of cRDSRxSignalProcessor (RDSProcess.cpp:168 ProcessNewRdsBit sequence, :312,355
 * DecodeRDS(uint16_t[4]) groups).  Bits are the differentially decoded data bits in arrival order.
 * Both calls synchronise with the device, run the integer block-sync / FEC state machine
 * (RDSProcess.cpp:272-431) on the host for new bits, and drain what they return. */
RFM_API int rfm_decoder_rds_take_groups(rfm_decoder* d, uint32_t stream, uint16_t* groups /* [max][4] */,
                                        uint32_t max_groups, uint32_t* n_groups);
RFM_API int rfm_decoder_rds_take_bits(rfm_decoder* d, uint32_t stream, uint8_t* bits, uint32_t max_bits,
                                      uint32_t* n_bits);
/* The UECP byte stream the add-on publishes on its RDS PID: every decoded group of the stream goes through the
 * stream's own group decoder (cRDSGroupDecoder::DecodeRDS, RDSGroupDecoder.cpp:166-272, see rfm_rdsgroup below) the
 * moment the block synchroniser delivers it, the frames are framed as cRadioReceiver::AddUECPDataFrame does
 * (RadioReceiver.cpp:387-414).  Independent of rfm_decoder_rds_take_groups: both see every group once. */
RFM_API int rfm_decoder_rds_take_uecp(rfm_decoder* d, uint32_t stream, uint8_t* out, uint32_t cap, uint32_t* n_bytes);

typedef struct rfm_stream_status
{
  int32_t stereo_detected;  /* cFmDecoder::StereoDetected, FmDecode.h:140 */
  float interface_level;    /* GetInterfaceLevel, FmDecode.h:155 */
  float baseband_level;     /* GetBasebandLevel, FmDecode.h:160 */
  float baseband_mean;      /* m_BasebandMean */
  float pilot_level;        /* GetPilotLevel, FmDecode.h:165 */
  float tuning_offset;      /* GetTuningOffset, FmDecode.h:146-150 */
} rfm_stream_status;
RFM_API int rfm_decoder_get_status(rfm_decoder* d, uint32_t stream, rfm_stream_status* out);

/* Derived constants / tables for known-answer tests against the reference constructors.
 * Same index list as oracle/ref_harness.cpp:ref_fm_constants / ref_fm_table. */
RFM_API int rfm_decoder_constants(const rfm_decoder* d, double* out, uint32_t max);
RFM_API int rfm_decoder_table(const rfm_decoder* d, int which, float* out, uint32_t max_floats, uint32_t* n);
/* The same, host-only (no device needed): the planner that restates the reference constructors
 * (cFmDecoder ctor FmDecode.cpp:237-314, cRDSRxSignalProcessor ctor RDSProcess.cpp:43-88).
 * table: 0 fine-tuner, 1 input Lanczos taps, 2 audio Lanczos taps, 3 RDS LP, 4 RDS matched filter,
 * 5 audio LP, 6 u8 -> float LUT (RTL_SDR_Source.cpp:207-211). */
RFM_API int rfm_plan_constants(const rfm_config* cfg, double* out, uint32_t max);
RFM_API int rfm_plan_table(const rfm_config* cfg, int which, float* out, uint32_t max_floats, uint32_t* n);

/* Per-kernel device timing for the roofline report: while on, every kernel launch is bracketed by CUDA events
 * on the stream it is launched on.  set_profiling() also clears the accumulated totals.  profile_read()
 * enumerates kernels: returns RFM_OK and fills name / total_ms / launches for index 0..k-1, 1 past the end
 * (index 0 synchronises and collects).  No reference counterpart (the reference only has commented-out
 * StartPerformance()/StopPerformance() hooks, DownConvert.cpp:418,487). */
RFM_API int rfm_decoder_set_profiling(rfm_decoder* d, int on);
/* A CUDA stream (cudaStream_t, owned by the decoder) on the FIR side of the decoder's SM partition -- an ordinary
 * non-blocking stream when rfm_config::lanes_sms leaves the decoder unpartitioned -- for the caller's own kernels that
 * produce the decoder's device input (rfm_downconvert / rfm_freqshift in front of rfm_decoder_process_cf32_device: the
 * composition of CRDSDownConvert::ProcessData and cFmDecoder::ProcessStream).  Work launched there never shares an SM
 * with the latency-bound lanes kernel (cPilotPhaseLock::Process and the other per-stream recurrences, FmDecode.cpp:149-216). */
RFM_API int rfm_decoder_companion_stream(rfm_decoder* d, void** stream);
RFM_API int rfm_decoder_profile_read(rfm_decoder* d, uint32_t index, char* name, uint32_t name_cap,
                                     double* total_ms, uint64_t* launches);

/* Telemetry of the time-parallel FM-demodulator PLL: number of 192-sample chunks (summed over streams) whose
 * speculative result had to be recomputed sequentially since the decoder was created (see DESIGN.md). */
RFM_API int rfm_decoder_demod_repairs(rfm_decoder* d, uint64_t* chunks);

/* Debug taps of the last block, copied to host (rows of n_streams).  name: demod_in baseband rawstereo
 * mono_rs stereo_rs lp rds_dec rds_lp rds_pll rds_mf.  Returns floats per stream in *n_floats. */
RFM_API int rfm_decoder_tap(rfm_decoder* d, const char* name, uint32_t stream, float* out, uint32_t max_floats,
                            uint32_t* n_floats);

/* ------------------------------------------------------------------------------------------------
 * cFreqShift (FreqShift.h:12-27, FreqShift.cpp:10-76), batched over rows: one NCO per row (stations of one
 * wideband capture, or independent streams).  Bug-compatible with the reference's x86 branch: float32 phase,
 * float32 increment float(K_2PI * f / Fs), never wrapped.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_freqshift rfm_freqshift;
/* cFreqShift(NcoFreq, InRate) per row -- FreqShift.cpp:10-16 */
RFM_API int rfm_freqshift_create(uint32_t rows, const float* nco_freq, float in_rate, uint32_t max_len, int device,
                                 rfm_freqshift** out);
RFM_API void rfm_freqshift_destroy(rfm_freqshift* f);
/* cFreqShift::Reset -- FreqShift.cpp:18-21 */
RFM_API int rfm_freqshift_reset(rfm_freqshift* f);
/* cFreqShift::Process(ComplexType* pInData, unsigned InLength), in place -- FreqShift.cpp:23-76; iq [rows][n][2] host */
RFM_API int rfm_freqshift_process_cf32(rfm_freqshift* f, float* iq, uint32_t n);
/* the same fused with cRtlSdrSource::ReadAsyncCB's u8 -> float conversion (RTL_SDR_Source.cpp:207-211): iq is one
 * shared capture [n][2] (shared_capture != 0: every row mixes the same samples with its own NCO) or [rows][n][2];
 * out [rows][n][2] float, host */
RFM_API int rfm_freqshift_process_u8(rfm_freqshift* f, const uint8_t* iq, int shared_capture, uint32_t n, float* out);
/* device pointers; mode 0: cf32 rows (d_out may alias d_in), 1: one shared u8 capture, 2: u8 rows; strides in samples */
RFM_API int rfm_freqshift_process_device(rfm_freqshift* f, int mode, const void* d_in, size_t in_stride, float* d_out,
                                         size_t out_stride, uint32_t n, void* cuda_stream);
/* Any rfm_iq_format, converted on the fly: iq is one shared capture [n] (shared_capture != 0) or [rows][n] samples of
 * `format`; out [rows][n][2] float.  Host form (blocking) and device form (enqueue only; strides in samples, in_stride is
 * ignored for a shared capture, d_in aligned to the sample size). */
RFM_API int rfm_freqshift_process_iq(rfm_freqshift* f, int format, int shared_capture, const void* iq, uint32_t n,
                                     float* out);
RFM_API int rfm_freqshift_process_iq_device(rfm_freqshift* f, int format, int shared_capture, const void* d_in,
                                            size_t in_stride, float* d_out, size_t out_stride, uint32_t n,
                                            void* cuda_stream);
/* IQ correction (rfm_iq_correction) of every input sample of every later process call, of every row; NULL = off (the
 * default).  Non-finite coefficients: RFM_ERR_INVALID. */
RFM_API int rfm_freqshift_set_iq_correction(rfm_freqshift* f, const rfm_iq_correction* c);

/* ------------------------------------------------------------------------------------------------
 * CRDSDownConvert (DownConvert.h:68-169, DownConvert.cpp:271-489), batched over rows: NCO_OSC mixer (the
 * amplitude-stabilised rotating vector of DownConvert.cpp:438-442, bit-exact) followed by the planned chain of
 * decimate-by-2 stages (half-bands HB11..HB51 of filtercoef.h:62-150, the fixed 11-tap stage, CIC3).
 * One row per station of a wideband capture (shared u8 input) or per independent stream.
 * n must be a multiple of 2^stages and long enough for every stage (RFM_ERR_UNSUPPORTED otherwise: the reference
 * itself mis-filters such calls, DownConvert.cpp:519-520,544-547).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_downconvert rfm_downconvert;
/* CRDSDownConvert() + SetDataRate(in_rate, max_bw) (wfm == 0, DownConvert.cpp:327-371) or SetWfmDataRate (wfm != 0,
 * :378-399) + SetFrequency(nco_freq[row]) (:311-320) */
RFM_API int rfm_downconvert_create(uint32_t rows, const float* nco_freq, float in_rate, float max_bw, int wfm,
                                   uint32_t max_len, int device, rfm_downconvert** out);
RFM_API void rfm_downconvert_destroy(rfm_downconvert* d);
/* the value SetDataRate / SetWfmDataRate return: in_rate / 2^stages */
RFM_API float rfm_downconvert_output_rate(const rfm_downconvert* d);
/* number of decimate-by-2 stages; taps[k] = length of stage k (3 = CIC3) */
RFM_API uint32_t rfm_downconvert_stages(const rfm_downconvert* d, uint32_t* taps, uint32_t max);
/* CRDSDownConvert::SetFrequency for every row (the carried oscillator phasors are kept) -- DownConvert.cpp:311-320 */
RFM_API int rfm_downconvert_set_frequency(rfm_downconvert* d, const float* nco_freq);
/* back to the freshly constructed state (m_Osc1 = 1 + 0j, empty delay lines) */
RFM_API int rfm_downconvert_reset(rfm_downconvert* d);
/* CRDSDownConvert::ProcessData(InLength, pInData, pOutData) -- DownConvert.cpp:412-489.  iq [rows][n][2] host (left
 * untouched; the reference scribbles its intermediate results over pInData), out [rows][n >> stages][2] host;
 * *n_out = the return value, n >> stages */
RFM_API int rfm_downconvert_process_cf32(rfm_downconvert* d, const float* iq, uint32_t n, float* out, uint32_t* n_out);
/* the same fused with cRtlSdrSource::ReadAsyncCB's u8 -> float conversion (RTL_SDR_Source.cpp:207-211); iq is one
 * shared capture [n][2] (shared_capture != 0) or [rows][n][2] */
RFM_API int rfm_downconvert_process_u8(rfm_downconvert* d, const uint8_t* iq, int shared_capture, uint32_t n, float* out,
                                       uint32_t* n_out);
/* Optional pre-mixer for phase-coherent blocks of a wideband capture: a cFreqShift that is Reset() every `period`
 * samples (FreqShift.cpp:18-21) repeats the same (cos, sin) sequence, so it is a lookup table: d_table [rows][row_stride]
 * float2 on the device, entry i = what cFreqShift::Process makes of the sample (1, 0) at position i after Reset()
 * (rfm_freqshift_process_* on a block of ones).  Every input sample is multiplied by its entry (the four products, one
 * subtraction, one addition of FreqShift.cpp:63-69) before CRDSDownConvert's own NCO.  The position starts at 0 when
 * the table is set or the converter reset and advances with the samples processed.  d_table == NULL switches it off. */
RFM_API int rfm_downconvert_set_premix(rfm_downconvert* d, const float* d_table, size_t row_stride, uint32_t period);
/* device pointers, enqueue only; mode 0: cf32 rows, 1: one shared u8 capture, 2: u8 rows; strides in samples */
RFM_API int rfm_downconvert_process_device(rfm_downconvert* d, int mode, const void* d_in, size_t in_stride, float* d_out,
                                           size_t out_stride, uint32_t n, uint32_t* n_out, void* cuda_stream);
/* Any rfm_iq_format, converted on the fly: iq is one shared capture [n] (shared_capture != 0) or [rows][n] samples of
 * `format`; out [rows][n >> stages][2] float.  Host form (blocking) and device form (enqueue only; strides in samples,
 * in_stride is ignored for a shared capture, d_in aligned to the sample size). */
RFM_API int rfm_downconvert_process_iq(rfm_downconvert* d, int format, int shared_capture, const void* iq, uint32_t n,
                                       float* out, uint32_t* n_out);
RFM_API int rfm_downconvert_process_iq_device(rfm_downconvert* d, int format, int shared_capture, const void* d_in,
                                              size_t in_stride, float* d_out, size_t out_stride, uint32_t n,
                                              uint32_t* n_out, void* cuda_stream);
/* IQ correction (rfm_iq_correction) of every input sample of every later process call, of every row, before the
 * pre-mix table and the NCO; NULL = off (the default).  Non-finite coefficients: RFM_ERR_INVALID. */
RFM_API int rfm_downconvert_set_iq_correction(rfm_downconvert* d, const rfm_iq_correction* c);
/* Phase-accumulator NCO pre-mixer, exact and parallel in time (DESIGN.md section 15; oracle/nco.py restates it).  In
 * the place of the pre-mix table: after the format conversion and the IQ correction, before CRDSDownConvert's own NCO
 * (normally at 0 Hz when this one is used).  Per row:
 *   word    d = (uint32_t)(int64_t) llround(nco_freq / (double)in_rate * 2^32), |nco_freq| <= in_rate / 2; the sign as
 *           for nco_freq of rfm_downconvert_create (-f brings a station at +f to 0 Hz)
 *   phase   sample i of a call: phi = (phi_start + i d) mod 2^32; phi_start = 0 after this call and after
 *           rfm_downconvert_reset, and advances by n d mod 2^32 with every call of n samples
 *   phasor  e = T0[phi >> 24] T1[(phi >> 16) & 255] T2[(phi >> 8) & 255], T_m[k] = exp(j 2 pi k / 2^(8 (m + 1))) as
 *           float(cos), float(sin) of a double angle; y = x e, every complex product the four products, one
 *           subtraction and one addition of the reference's mixers, each rounded on its own.
 * Error against exp(j 2 pi phi / 2^32): about -133 dBc; frequency within in_rate / 2^33.  nco_freq [rows] Hz; NULL
 * switches it off.  RFM_ERR_INVALID for a non-finite or out-of-range frequency, or while a pre-mix table is set
 * (rfm_downconvert_set_premix likewise refuses a table while the NCO is set). */
RFM_API int rfm_downconvert_set_nco(rfm_downconvert* d, const double* nco_freq);

/* ------------------------------------------------------------------------------------------------
 * cDownsampleFilter (DownConvert.h:21-60, DownConvert.cpp:58-256), batched over rows: Lanczos-windowed sinc FIR with
 * decimation, in the two forms the chain uses -- complex input + integer factor (m_ReSampleInput, FmDecode.cpp:257-261)
 * and real input + fractional factor (m_ReSampleMono / m_ReSampleStereo, :263-273) -- plus real input + integer
 * factor (DownConvert.cpp:164-192; no caller in the reference).  Complex + fractional (an endless loop in the
 * reference) and calls shorter than the filter order return RFM_ERR_UNSUPPORTED.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_downsample rfm_downsample;
/* cDownsampleFilter(filter_order, cutoff, downsample, integer_factor) -- DownConvert.cpp:63-81 */
RFM_API int rfm_downsample_create(uint32_t rows, uint32_t filter_order, double cutoff, double downsample,
                                  int integer_factor, uint32_t max_len, int device, rfm_downsample** out);
RFM_API void rfm_downsample_destroy(rfm_downsample* f);
/* cDownsampleFilter::Reset -- DownConvert.cpp:90-96 */
RFM_API int rfm_downsample_reset(rfm_downsample* f);
/* m_coeff: filter_order + 2 entries (MakeLanczosCoeff, DownConvert.cpp:18-56) */
RFM_API int rfm_downsample_coefficients(const rfm_downsample* f, float* out, uint32_t max, uint32_t* n);
/* upper bound of the outputs of an n-sample call (size of the caller's output rows) */
RFM_API uint32_t rfm_downsample_max_outputs(const rfm_downsample* f, uint32_t n);
/* unsigned Process(const ComplexType*, ComplexType*, unsigned) -- DownConvert.cpp:98-154; in [rows][n][2] host,
 * out [rows][*n_out][2] host (rows packed back to back); *n_out = the return value */
RFM_API int rfm_downsample_process_complex(rfm_downsample* f, const float* in, float* out, uint32_t n, uint32_t* n_out);
/* unsigned Process(const RealType*, RealType*, unsigned) -- DownConvert.cpp:156-256 (integer branch :164-192,
 * fractional branch :195-233, whichever the object was created with) */
RFM_API int rfm_downsample_process_real(rfm_downsample* f, const float* in, float* out, uint32_t n, uint32_t* n_out);
/* device rows, enqueue only; strides in samples */
RFM_API int rfm_downsample_process_complex_device(rfm_downsample* f, const float* d_in, size_t in_stride, float* d_out,
                                                  size_t out_stride, uint32_t n, uint32_t* n_out, void* cuda_stream);
RFM_API int rfm_downsample_process_real_device(rfm_downsample* f, const float* d_in, size_t in_stride, float* d_out,
                                               size_t out_stride, uint32_t n, uint32_t* n_out, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * cIirFilter (IirFilter.h:12-36, IirFilter.cpp:11-105), batched over rows (one independent biquad per row, all with
 * the same coefficients).  type: 0 ftLP, 1 ftHP, 2 ftBP, 3 ftBR (IirFilter.h:15).  Buffers are filtered in place.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_iir rfm_iir;
RFM_API int rfm_iir_create(uint32_t rows, uint32_t max_len, int device, rfm_iir** out);
RFM_API void rfm_iir_destroy(rfm_iir* f);
/* cIirFilter::Init -- IirFilter.cpp:11-60.  Clears the delays; an unknown type returns RFM_ERR_INVALID (Init returns
 * false) and keeps the previous coefficients */
RFM_API int rfm_iir_init(rfm_iir* f, int type, float F0Freq, float FilterQ, float SampleRate);
/* m_A1, m_A2, m_B0, m_B1, m_B2 */
RFM_API int rfm_iir_coefficients(const rfm_iir* f, float* out5);
/* cIirFilter::Process(RealType*, n) :78-87 / Process(ComplexType*, n) :62-76 / ProcessTwo(RealType*, RealType*, n) :89-105;
 * host buffers [rows][n] ([rows][n][2] for complex) */
RFM_API int rfm_iir_process_real(rfm_iir* f, float* buf, uint32_t n);
RFM_API int rfm_iir_process_complex(rfm_iir* f, float* buf, uint32_t n);
RFM_API int rfm_iir_process_two(rfm_iir* f, float* a, float* b, uint32_t n);
/* device pointers, enqueue only; mode 0 real, 1 complex, 2 two buffers; stride in elements (complex: in samples) */
RFM_API int rfm_iir_process_device(rfm_iir* f, int mode, float* d_a, float* d_b, size_t stride, uint32_t n,
                                   void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * cFirFilter (FirFilter.h:17-60, FirFilter.cpp), batched over rows: Kaiser low-/high-pass design or constant taps, the
 * circular delay line with its rotating summation start (the sum of a given output begins at the tap the reference's
 * m_State points at, so the rounding sequence is the reference's).  Buffers are filtered in place.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_fir rfm_fir;
RFM_API int rfm_fir_create(uint32_t rows, uint32_t max_len, int device, rfm_fir** out);
RFM_API void rfm_fir_destroy(rfm_fir* f);
/* cFirFilter::InitLPFilter(NumTaps, Scale, Astop, Fpass, Fstop, Fsamprate) -- FirFilter.cpp:78-148; *ntaps = its
 * return value (the tap count, computed from the specification when NumTaps == 0) */
RFM_API int rfm_fir_init_lp(rfm_fir* f, uint32_t NumTaps, float Scale, float Astop, float Fpass, float Fstop, float Fs,
                            uint32_t* ntaps);
/* cFirFilter::InitHPFilter(NumTaps, Scale, Astop, Fpass, Fstop, Fsamprate) -- FirFilter.cpp:195-264 (no caller in the
 * reference; odd tap count, at most 73 unless forced) */
RFM_API int rfm_fir_init_hp(rfm_fir* f, uint32_t NumTaps, float Scale, float Astop, float Fpass, float Fstop, float Fs,
                            uint32_t* ntaps);
/* the Kaiser designs alone, host only (no device): kind 0 = InitLPFilter's taps, 1 = InitHPFilter's; *n = tap count */
RFM_API int rfm_fir_design(int kind, uint32_t NumTaps, float Scale, float Astop, float Fpass, float Fstop, float Fs,
                           float* out, uint32_t max, uint32_t* n);
/* cFirFilter::InitConstFir(NumTaps, const RealType* pCoef, Fsamprate) -- FirFilter.cpp:302-320 */
RFM_API int rfm_fir_init_const(rfm_fir* f, uint32_t ntaps, const float* coef, float Fs);
RFM_API int rfm_fir_taps(const rfm_fir* f, float* out, uint32_t max, uint32_t* n);
/* cFirFilter::Process(RealType*, n) :360-377 / Process(ComplexType*, n) :330-350 / ProcessTwo :387-413 */
RFM_API int rfm_fir_process_real(rfm_fir* f, float* buf, uint32_t n);
RFM_API int rfm_fir_process_complex(rfm_fir* f, float* buf, uint32_t n);
RFM_API int rfm_fir_process_two(rfm_fir* f, float* a, float* b, uint32_t n);
RFM_API int rfm_fir_process_device(rfm_fir* f, int mode, float* d_a, float* d_b, size_t stride, uint32_t n,
                                   void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * cRDSRxSignalProcessor (RDSProcess.h:56-110, RDSProcess.cpp:43-431), batched over rows: demodulated FM baseband in,
 * RDS bits and groups out.  Float part on the device, block synchronisation / FEC on the host (as rfm_rdssync).
 * n must be a multiple of 2^stages of the RDS decimation chain (RFM_ERR_UNSUPPORTED otherwise, see rfm_downconvert).
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_rdsproc rfm_rdsproc;
/* cRDSRxSignalProcessor(proc, SampleRate) -- RDSProcess.cpp:43-88 */
RFM_API int rfm_rdsproc_create(uint32_t rows, float sample_rate, uint32_t max_len, int device, rfm_rdsproc** out);
RFM_API void rfm_rdsproc_destroy(rfm_rdsproc* r);
/* m_ProcessRate */
RFM_API float rfm_rdsproc_process_rate(const rfm_rdsproc* r);
/* cRDSRxSignalProcessor::Reset -- RDSProcess.cpp:90-118 */
RFM_API int rfm_rdsproc_reset(rfm_rdsproc* r);
/* cRDSRxSignalProcessor::Process(const RealType* inputStream, unsigned inLength) -- RDSProcess.cpp:120-180;
 * baseband [rows][n] host */
RFM_API int rfm_rdsproc_process(rfm_rdsproc* r, const float* baseband, uint32_t n);
/* device rows [rows][stride], enqueue only (bits are fetched by the take calls) */
RFM_API int rfm_rdsproc_process_device(rfm_rdsproc* r, const float* d_bb, size_t stride, uint32_t n, void* cuda_stream);
/* the arguments of successive ProcessNewRdsBit calls (RDSProcess.cpp:168) / the groups handed to DecodeRDS (:312,355) */
RFM_API int rfm_rdsproc_take_bits(rfm_rdsproc* r, uint32_t row, uint8_t* bits, uint32_t max_bits, uint32_t* n_bits);
RFM_API int rfm_rdsproc_take_groups(rfm_rdsproc* r, uint32_t row, uint16_t* groups, uint32_t max_groups,
                                    uint32_t* n_groups);

/* Test hooks (no reference counterpart): evaluate one of the scalar building blocks of the kernels on the DEVICE for
 * n host operands; out2 receives two floats per element.  op: 0 rfm_sincos (sin, cos) 1 sincos fast core
 * 2 sincos generic 3 atan2f(a, b) 4 branch-free atan2f (+flag) 5 atan2f generic 6 branch-free a / b (+flag)
 * 7 __fdiv_rn 8 / 9 branch-free demod / pilot phase wrap (+flag) 10 both exact wraps 11 RDS arctan2 approximation
 * (RDSProcess.cpp:187-217) 12 fmodf 13 NCO_OSC gain (float form, double form).  rfm_div_selftest: branch-free division vs __fdiv_rn over `pairs` random
 * operand pairs generated on the device. */
RFM_API int rfm_math_probe(int op, const float* a, const float* b, float* out2, uint32_t n);
RFM_API int rfm_div_selftest(uint64_t seed, uint64_t pairs, uint64_t* mismatches, uint64_t* tested);

/* ------------------------------------------------------------------------------------------------
 * RDS block synchronisation / FEC on explicit bits (host integer code, RDSProcess.cpp:272-431)
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_rdssync rfm_rdssync;
RFM_API int rfm_rdssync_create(rfm_rdssync** out);
RFM_API void rfm_rdssync_destroy(rfm_rdssync* s);
RFM_API void rfm_rdssync_reset(rfm_rdssync* s);
RFM_API int rfm_rdssync_push_bits(rfm_rdssync* s, const uint8_t* bits, uint32_t n);
RFM_API int rfm_rdssync_take_groups(rfm_rdssync* s, uint16_t* groups, uint32_t max_groups, uint32_t* n_groups);
/* cRDSRxSignalProcessor::CheckBlock, RDSProcess.cpp:377-431 */
RFM_API uint32_t rfm_rds_check_block(uint32_t word26, uint32_t offset_syndrome, int use_fec, uint32_t* corrected);

/* ------------------------------------------------------------------------------------------------
 * RDS groups -> UECP frames (host integer code): cRDSGroupDecoder(cRadioReceiver*), Reset(), DecodeRDS(uint16_t*)
 * (RDSGroupDecoder.h:24-31, RDSGroupDecoder.cpp:136-1001 with the reference's default build macros).
 * The callbacks are the three calls the reference makes on its cRadioReceiver from inside DecodeRDS
 * (RadioReceiver.h:77,80,115); any of them may be NULL:
 *   add_uecp_frame    NULL: frames collect inside the object in the transport framing of
 *                     cRadioReceiver::AddUECPDataFrame (0xFE, byte stuffing, 0xFF) -> rfm_rdsgroup_take_uecp
 *   set_channel_name  NULL: every name is accepted (RadioReceiver.cpp:600-612 without a settings dialog) and kept
 *                     -> rfm_rdsgroup_channel_name
 *   is_setting_active NULL: never active
 * Members the reference leaves uninitialised (m_PTY, m_DI_Finished, m_RadioText_ABFlag, m_PTYN_ABFlag,
 * m_UECPDataFrameSeqCnt) start at zero here; its function-static PS buffer is per object.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_rdsgroup rfm_rdsgroup;
typedef struct rfm_rdsgroup_callbacks
{
  void* user;
  int (*add_uecp_frame)(void* user, const uint8_t* frame, uint32_t len);
  int (*set_channel_name)(void* user, const char* name8); /* nonzero: accepted */
  int (*is_setting_active)(void* user);
} rfm_rdsgroup_callbacks;
RFM_API int rfm_rdsgroup_create(const rfm_rdsgroup_callbacks* cb /* may be NULL */, rfm_rdsgroup** out);
RFM_API void rfm_rdsgroup_destroy(rfm_rdsgroup* g);
RFM_API void rfm_rdsgroup_reset(rfm_rdsgroup* g);
RFM_API int rfm_rdsgroup_decode(rfm_rdsgroup* g, const uint16_t* blocks /* [n_groups][4] */, uint32_t n_groups);
RFM_API int rfm_rdsgroup_take_uecp(rfm_rdsgroup* g, uint8_t* out, uint32_t cap, uint32_t* n_bytes);
RFM_API int rfm_rdsgroup_channel_name(const rfm_rdsgroup* g, char out[9]);
/* cRadioReceiver::AddUECPDataFrame's framing alone; returns the framed length (written only when it fits cap) */
RFM_API uint32_t rfm_uecp_stuff_frame(const uint8_t* frame, uint32_t len, uint8_t* out, uint32_t cap);

/* ------------------------------------------------------------------------------------------------
 * The caller of the hot path: IQ block queue + packetiser of cRadioReceiver (RadioReceiver.cpp:420-542), one
 * programme.  Source thread: rfm_demux_write_u8 (WriteDataBuffer, the block stays u8 and goes to pinned memory) /
 * rfm_demux_end (EndDataBuffer).  Demux thread: rfm_demux_read (DemuxRead) hands out, in the reference's order, the
 * stream-change packet, then for every block its audio packet (stream id 1: interleaved float L,R, pts / duration in
 * STREAM_TIME_BASE = 1e6 units, pts starting at 1e6) followed by a UECP packet (stream id 2, pts of the NEXT audio
 * packet) when the block's RDS groups produced frames.  `data` stays valid until the next packet of the same stream
 * id is read.  The block after the one just handed out is decoded ahead when it is already queued.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_demux rfm_demux;
#define RFM_DEMUX_STREAMCHANGE (-11) /* DEMUX_SPECIALID_STREAMCHANGE */
#define RFM_DEMUX_END 1              /* rfm_demux_read: end marked and every block handed out (reference: nullptr) */
typedef struct rfm_demux_packet
{
  int32_t stream_id;    /* 1 audio, 2 UECP, RFM_DEMUX_STREAMCHANGE */
  uint32_t size_bytes;  /* iSize */
  double pts, duration;
  const void* data;     /* pData */
} rfm_demux_packet;
RFM_API int rfm_demux_create(const rfm_config* cfg /* n_streams is taken as 1 */, rfm_demux** out);
RFM_API void rfm_demux_destroy(rfm_demux* m);
RFM_API rfm_decoder* rfm_demux_decoder(rfm_demux* m); /* the cFmDecoder behind it (getters, Reset) */
RFM_API int rfm_demux_write_u8(rfm_demux* m, const uint8_t* iq, uint32_t n);
RFM_API int rfm_demux_end(rfm_demux* m);
RFM_API uint64_t rfm_demux_queued_samples(rfm_demux* m); /* SourceQueuedSamples */
RFM_API void rfm_demux_set_stream_change(rfm_demux* m);  /* SetStreamChange, RadioReceiver.h:83 */
RFM_API int rfm_demux_read(rfm_demux* m, rfm_demux_packet* pkt);
RFM_API float rfm_demux_audio_level(const rfm_demux* m);  /* m_AudioLevel, RadioReceiver.cpp:528-529 */
/* The source side of cRtlSdrSource (SURVEY.md 8f N4) without librtlsdr: its block-length rule (clamp to 4096 .. 2^20,
 * multiple of 4096; RTL_SDR_Source.cpp:124-126) and its async read callback (RTL_SDR_Source.cpp:196-213) with the
 * signature of rtlsdr_read_async_cb_t -- pass it to rtlsdr_read_async with ctx = the rfm_demux and
 * buf_len = 2 * block length.  Buffers of any other length are dropped and counted, as the reference drops them. */
RFM_API uint32_t rfm_source_block_length(uint32_t requested);
RFM_API int rfm_demux_set_source_block_length(rfm_demux* m, uint32_t requested);
RFM_API void rfm_demux_source_cb(unsigned char* buf, uint32_t len, void* ctx);
RFM_API uint64_t rfm_demux_short_reads(rfm_demux* m);

/* cRtlSdrSource itself (RTL_SDR_Source.h:21-86, RTL_SDR_Source.cpp:27-256): librtlsdr bound at run time with dlopen
 * (`library` = path or soname, NULL = librtlsdr.so.0 / librtlsdr.so; RFM_ERR_UNSUPPORTED when it cannot be loaded,
 * RFM_ERR_NO_DEVICE when rtlsdr_open fails).  open = cRtlSdrSource::Open; configure = Configure (sample rate, centre
 * frequency, manual gain in 0.1 dB or INT_MIN for automatic, RTL AGC, block length by the rule above,
 * rtlsdr_reset_buffer) and starts the reader thread (Process: rtlsdr_read_async with 15 buffers of 2 * block bytes,
 * up to five re-configure attempts after a failed read, EndDataBuffer at the end); every full block is queued raw into
 * `demux` by rfm_demux_source_cb; close = Close (rtlsdr_cancel_async, join) + rtlsdr_close. */
typedef struct rfm_rtlsdr rfm_rtlsdr;
RFM_API int rfm_rtlsdr_device_count(const char* library);
RFM_API int rfm_rtlsdr_open(rfm_demux* demux, const char* library, int dev_index, rfm_rtlsdr** out);
RFM_API int rfm_rtlsdr_configure(rfm_rtlsdr* s, uint32_t sample_rate, uint32_t frequency, int tuner_gain,
                                 int block_length, int agcmode);
RFM_API void rfm_rtlsdr_close(rfm_rtlsdr* s);
RFM_API uint32_t rfm_rtlsdr_get_sample_rate(rfm_rtlsdr* s);   /* GetSampleRate */
RFM_API uint32_t rfm_rtlsdr_get_frequency(rfm_rtlsdr* s);     /* GetFrequency */
RFM_API void rfm_rtlsdr_set_frequency(rfm_rtlsdr* s, uint32_t freq);
RFM_API int rfm_rtlsdr_get_tuner_gain(rfm_rtlsdr* s);         /* GetTunerGain */
RFM_API uint32_t rfm_rtlsdr_block_length(const rfm_rtlsdr* s); /* m_BlockLength */
RFM_API uint32_t rfm_rtlsdr_restarts(const rfm_rtlsdr* s);
RFM_API const char* rfm_rtlsdr_error(const rfm_rtlsdr* s);    /* error() */
/* GetSignalStatus(float&, float&, bool&), RadioReceiver.cpp:544-556: levels in dB */
RFM_API int rfm_demux_signal_status(rfm_demux* m, float* interface_level_db, float* audio_level_db, int* stereo);

/* ------------------------------------------------------------------------------------------------
 * Band scan of one wideband capture: the add-on's tuner auto-scan (ChannelSettings.cpp:96-147: retune one frequency,
 * wait, check cFmDecoder::StereoDetected) generalised to every channel of a capture in one pass.
 *   spectrum   Welch average over N = 4096 periodic-Hann segments, hop N/2, of the capture converted to float as
 *              rfm_iq_format says (u8: float(u / 127.5 - 1), RTL_SDR_Source.cpp:207-211): P[k] = sum_s |X_s[k]|^2 / (S N sum w^2), so sum_k P is the mean power of
 *              the windowed signal (a complex tone of modulus 1 is 0 dBFS).  Centred: index k <-> (k - N/2) Fs / N Hz.
 *              Independent of the device, its SM count and any SM partition (fixed work split, no atomics).
 *   channels   raster point f_j = raster_first + j raster_step owns the bins with f_j - step/2 <= f < f_j + step/2;
 *              C_j = sum of its bins' P in double, in bin order.  floor = the sorted C at index (count - 1) / 4.
 *   candidate  C_j >= floor * 10^(min_snr_db / 10), C_j > C_{j-1} (when j-1 exists), C_j >= C_{j+1} (when j+1 exists).
 *   stations   every candidate confirmed with the reference's receiver over every whole call of the capture: rows of
 *              rfm_downconvert (CRDSDownConvert::SetFrequency(-f_j) + SetWfmDataRate(Fs, 100 kHz)) into one
 *              rfm_decoder (cFmDecoder(rate, 0, 48000, 15000, 1)); one call = 16000 baseband samples
 *              (16000 << stages capture samples).  PS is what cRDSGroupDecoder hands to SetChannelName for the groups.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rfm_scan rfm_scan;
typedef struct rfm_scan_config
{
  double sample_rate;                 /* capture rate, Hz */
  double raster_first, raster_step;   /* Hz from the capture centre; step >= 4 Fs / 4096 */
  uint32_t raster_count;              /* 1 .. 4096; every |f_j| + 100 kHz <= Fs / 2 */
  double min_snr_db;                  /* default 10 */
  int32_t device;                     /* -1 = current */
} rfm_scan_config;
typedef struct rfm_scan_station
{
  double freq;                        /* raster frequency, Hz from the capture centre */
  float power_dbfs, snr_db;           /* 10 log10 C_j, 10 log10 (C_j / floor) */
  int32_t stereo_detected;            /* rfm_stream_status after the last call */
  float pilot_level, interface_level, baseband_level;
  uint32_t rds_groups;                /* groups delivered by the block synchroniser */
  int32_t pi;                         /* most frequent block A, ties to the first seen; -1: no group */
  char ps[9];                         /* "" if no name was published */
} rfm_scan_station;
/* Defaults: 2.4 MS/s (the add-on's RTL-SDR rate), 100 kHz raster over +-1.1 MHz, 10 dB, current device. */
RFM_API void rfm_scan_config_default(rfm_scan_config* cfg);
/* Validates the raster (RFM_ERR_INVALID: step < 4 Fs / N, count outside 1 .. N, a channel with |f_j| + 100 kHz > Fs/2,
 * a rate whose WFM decimation chain has no stage) before touching a device. */
RFM_API int rfm_scan_create(const rfm_scan_config* cfg, rfm_scan** out);
RFM_API void rfm_scan_destroy(rfm_scan* s);
/* Whole capture of n samples of `format` (rfm_iq_format) in host memory (copied with cudaMemcpyAsync) or device memory
 * (complete before the call, aligned to the sample size: 2 / 2 / 4 / 8 bytes); n >= one call (RFM_ERR_INVALID
 * otherwise, as for an unknown format).  Blocking.  Zero candidates: no receiver is created and the scan has 0
 * stations.  A spectrum with a non-finite bin -- a NaN or Inf sample, a NaN dc from the mode-1 estimate, or a capture
 * large enough to overflow the float32 FFT (a coherent tone from |x| of about 1e15: 32 segments of |X|^2 per sum) --
 * has no floor and no candidates: RFM_ERR_INVALID, the bin in rfm_last_error(), before any decision; the handle keeps
 * no result and stays usable. */
RFM_API int rfm_scan_run(rfm_scan* s, int format, const void* iq, uint64_t n, int iq_on_device);
/* rfm_scan_run(s, RFM_IQ_U8, iq, n, iq_on_device) */
RFM_API int rfm_scan_run_u8(rfm_scan* s, const uint8_t* iq, uint64_t n, int iq_on_device);
RFM_API int rfm_scan_spectrum(rfm_scan* s, float* psd, uint32_t max, uint32_t* n_bins);   /* N floats, centred */
RFM_API int rfm_scan_channel_power(rfm_scan* s, double* out, uint32_t max);              /* C_j, linear */
RFM_API int rfm_scan_stations(rfm_scan* s, rfm_scan_station* out, uint32_t max, uint32_t* n);
/* Device time of the last run's two stages (CUDA events): the spectrum kernels, and the confirmation from the first
 * front-end launch to the end of the last demodulator call (0 without candidates). */
RFM_API int rfm_scan_timing(rfm_scan* s, double* spectrum_ms, double* confirm_ms);
/* IQ correction of later runs (rfm_iq_correction): mode 0 off (the default), 1 estimate from each run's capture (one
 * statistics pass before the spectrum; the capture must then hold at most 2^32 samples), 2 use `fixed` (copied).  The
 * spectrum is that of the corrected samples and the confirmation's rfm_downconvert rows carry the same correction.
 * RFM_ERR_INVALID for an unknown mode, a NULL `fixed` with mode 2 or non-finite coefficients. */
RFM_API int rfm_scan_set_iq_correction(rfm_scan* s, int mode, const rfm_iq_correction* fixed);
/* What the last run applied; mode 0: {0, 0, 1, 0, imbalance_valid = 0} */
RFM_API int rfm_scan_iq_correction(rfm_scan* s, rfm_iq_correction* out);
/* Mixer of the confirmation's rfm_downconvert rows in later runs: RFM_SCAN_MIXER_OSC (the default) sets each row's
 * CRDSDownConvert NCO to -f_j; RFM_SCAN_MIXER_NCO creates the rows at 0 Hz and sets rfm_downconvert_set_nco(-f_j).
 * RFM_ERR_INVALID for another value. */
enum { RFM_SCAN_MIXER_OSC = 0, RFM_SCAN_MIXER_NCO = 1 };
RFM_API int rfm_scan_set_mixer(rfm_scan* s, int mixer);

#ifdef __cplusplus
}
#endif
#endif /* RADIOFM_B200_H */
