// tests/cpp/host_nco_driver.cpp -- the phasor NCO through the C ABI alone (include/radiofm_b200.h): scan a u8 capture
// with the "nco" confirmation (rfm_scan_set_mixer), then decode the strongest station with an rfm_downconvert created at
// 0 Hz and moved by rfm_downconvert_set_nco(-f), feeding rfm_decoder_process_iq_device, and print what each step reports.
// It also checks the refusals of rfm_downconvert_set_nco and rfm_scan_set_mixer.
//   usage: host_nco_driver <capture_u8.bin> <fs> <raster_first> <raster_step> <raster_count>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "radiofm_b200.h"

static int Fail(const char* what, int rc)
{
  fprintf(stderr, "%s: error %d: %s\n", what, rc, rfm_last_error());
  return 1;
}

int main(int argc, char** argv)
{
  if (argc != 6)
  {
    fprintf(stderr, "usage: %s capture_u8.bin fs raster_first raster_step raster_count\n", argv[0]);
    return 2;
  }
  FILE* f = fopen(argv[1], "rb");
  if (!f)
  {
    perror(argv[1]);
    return 1;
  }
  std::vector<uint8_t> cap;
  uint8_t buf[1 << 16];
  size_t k;
  while ((k = fread(buf, 1, sizeof(buf), f)) > 0)
    cap.insert(cap.end(), buf, buf + k);
  fclose(f);
  const uint64_t n = cap.size() / 2;

  // 1. scan with the phasor NCO in front of rows at 0 Hz
  rfm_scan_config cfg;
  rfm_scan_config_default(&cfg);
  cfg.sample_rate = atof(argv[2]);
  cfg.raster_first = atof(argv[3]);
  cfg.raster_step = atof(argv[4]);
  cfg.raster_count = (uint32_t)atoi(argv[5]);
  rfm_scan* s = nullptr;
  int rc = rfm_scan_create(&cfg, &s);
  if (rc == RFM_OK && rfm_scan_set_mixer(s, 2) != RFM_ERR_INVALID)
    return Fail("rfm_scan_set_mixer accepted mixer 2", RFM_ERR_INVALID);
  if (rc == RFM_OK)
    rc = rfm_scan_set_mixer(s, RFM_SCAN_MIXER_NCO);
  if (rc == RFM_OK)
    rc = rfm_scan_run(s, RFM_IQ_U8, cap.data(), n, 0);
  std::vector<rfm_scan_station> st(cfg.raster_count);
  uint32_t ns = 0;
  if (rc == RFM_OK)
    rc = rfm_scan_stations(s, st.data(), (uint32_t)st.size(), &ns);
  rfm_scan_destroy(s);
  if (rc != RFM_OK)
    return Fail("rfm_scan", rc);
  printf("scan: %u stations\n", ns);
  for (uint32_t i = 0; i < ns; ++i)
    printf("station: offset_hz=%.0f dBFS=%.2f stereo=%d pi=%X ps=%s\n", st[i].freq, st[i].power_dbfs,
           st[i].stereo_detected, (unsigned)st[i].pi, st[i].ps);
  if (ns == 0)
    return 1;
  uint32_t best = 0;
  for (uint32_t i = 1; i < ns; ++i)
    if (st[i].power_dbfs > st[best].power_dbfs)
      best = i;

  // 2. front end at 0 Hz behind the NCO, then the decoder on device buffers
  const float zero = 0.0f;
  rfm_downconvert* dc = nullptr;
  rc = rfm_downconvert_create(1, &zero, (float)cfg.sample_rate, 100000.0f, 1, 1u << 22, -1, &dc);
  if (rc != RFM_OK)
    return Fail("rfm_downconvert_create", rc);
  const double too_far = 0.5 * cfg.sample_rate * (1.0 + 1e-9), not_finite = NAN;
  if (rfm_downconvert_set_nco(dc, &too_far) != RFM_ERR_INVALID || rfm_downconvert_set_nco(dc, &not_finite) != RFM_ERR_INVALID)
    return Fail("rfm_downconvert_set_nco accepted an invalid frequency", RFM_ERR_INVALID);
  const double nco = -st[best].freq;
  rc = rfm_downconvert_set_nco(dc, &nco);
  if (rc != RFM_OK)
    return Fail("rfm_downconvert_set_nco", rc);
  printf("refusals: ok\n");
  uint32_t taps[16];
  const uint32_t stages = rfm_downconvert_stages(dc, taps, 16);
  const uint32_t n_call = 16000u << stages;
  const uint64_t calls = n / n_call;
  std::vector<float> bb(2 * (size_t)(calls * 16000));
  for (uint64_t c = 0; c < calls; ++c)
  {
    uint32_t m = 0;
    rc = rfm_downconvert_process_iq(dc, RFM_IQ_U8, 1, cap.data() + 2 * c * n_call, n_call, bb.data() + 2 * c * 16000, &m);
    if (rc != RFM_OK || m != 16000)
      return Fail("rfm_downconvert_process_iq", rc);
  }
  const float rate = rfm_downconvert_output_rate(dc);
  rfm_downconvert_destroy(dc);
  rfm_config c;
  rfm_config_default(&c);
  c.sample_rate_if = rate;
  c.tuning_offset = 0.0;
  c.downsample = 1;
  c.n_streams = 1;
  c.max_block_len = 16000;
  c.n_groups = 1;
  rfm_decoder* d = nullptr;
  rc = rfm_decoder_create(&c, &d);
  if (rc != RFM_OK)
    return Fail("rfm_decoder_create", rc);
  const uint32_t stride = (rfm_decoder_max_audio_floats(d, 16000) + 3) & ~1u;
  float *d_bb = nullptr, *d_audio = nullptr;
  if (cudaMalloc(&d_bb, 16000 * 8) != cudaSuccess || cudaMalloc(&d_audio, (size_t)stride * 4) != cudaSuccess)
    return Fail("cudaMalloc", RFM_ERR_CUDA);
  for (uint64_t k2 = 0; k2 < calls; ++k2)
  {
    uint32_t na = 0;
    if (cudaMemcpyAsync(d_bb, bb.data() + 2 * k2 * 16000, 16000 * 8, cudaMemcpyHostToDevice, 0) != cudaSuccess)
      return Fail("cudaMemcpyAsync", RFM_ERR_CUDA);
    rc = rfm_decoder_process_iq_device(d, RFM_IQ_CF32, d_bb, 16000, 16000, d_audio, stride, &na, nullptr);
    if (rc == RFM_OK)
      rc = rfm_decoder_synchronize(d);
    if (rc != RFM_OK)
      return Fail("rfm_decoder_process_iq_device", rc);
  }
  rfm_stream_status ss;
  rc = rfm_decoder_get_status(d, 0, &ss);
  uint16_t groups[4 * 4096];
  uint32_t ng = 0;
  if (rc == RFM_OK)
    rc = rfm_decoder_rds_take_groups(d, 0, groups, 4096, &ng);
  if (rc != RFM_OK)
    return Fail("rfm_decoder status", rc);
  char ps[9] = "";
  rfm_rdsgroup* g = nullptr;
  if (rfm_rdsgroup_create(nullptr, &g) == RFM_OK && rfm_rdsgroup_decode(g, groups, ng) == RFM_OK)
    rfm_rdsgroup_channel_name(g, ps);
  rfm_rdsgroup_destroy(g);
  printf("decoded: offset_hz=%.0f stereo=%d groups=%u pi=%X ps=%s\n", st[best].freq, ss.stereo_detected, ng,
         ng ? (unsigned)groups[0] : 0u, ps);
  cudaFree(d_bb);
  cudaFree(d_audio);
  rfm_decoder_destroy(d);
  return 0;
}
