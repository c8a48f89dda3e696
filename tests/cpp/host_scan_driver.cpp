// tests/cpp/host_scan_driver.cpp -- a band scan through the C ABI alone (include/radiofm_b200.h, rfm_scan_*): reads a
// capture file (u8 I,Q pairs), scans it, prints the station table and writes it as raw rfm_scan_station records.
//   usage: host_scan_driver <capture_u8.bin> <fs> <raster_first> <raster_step> <raster_count> <stations_out.bin>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "radiofm_b200.h"

int main(int argc, char** argv)
{
  if (argc != 7)
  {
    fprintf(stderr, "usage: %s capture_u8.bin fs raster_first raster_step raster_count stations_out.bin\n", argv[0]);
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

  rfm_scan_config cfg;
  rfm_scan_config_default(&cfg);
  cfg.sample_rate = atof(argv[2]);
  cfg.raster_first = atof(argv[3]);
  cfg.raster_step = atof(argv[4]);
  cfg.raster_count = (uint32_t)atoi(argv[5]);
  rfm_scan* s = nullptr;
  int rc = rfm_scan_create(&cfg, &s);
  if (rc == RFM_OK)
    rc = rfm_scan_run_u8(s, cap.data(), cap.size() / 2, 0);
  std::vector<rfm_scan_station> st(cfg.raster_count);
  uint32_t n = 0;
  if (rc == RFM_OK)
    rc = rfm_scan_stations(s, st.data(), (uint32_t)st.size(), &n);
  if (rc != RFM_OK)
  {
    fprintf(stderr, "rfm_scan: error %d: %s\n", rc, rfm_last_error());
    rfm_scan_destroy(s);
    return 1;
  }
  printf("%12s %8s %7s %6s %6s %6s %8s\n", "offset_hz", "dBFS", "snr_dB", "stereo", "groups", "pi", "ps");
  for (uint32_t i = 0; i < n; ++i)
    printf("%12.0f %8.2f %7.2f %6d %6u %6X %8s\n", st[i].freq, st[i].power_dbfs, st[i].snr_db, st[i].stereo_detected,
           st[i].rds_groups, st[i].pi < 0 ? 0u : (unsigned)st[i].pi, st[i].ps);
  FILE* o = fopen(argv[6], "wb");
  if (!o || (n && fwrite(st.data(), sizeof(rfm_scan_station), n, o) != n))
  {
    perror(argv[6]);
    rfm_scan_destroy(s);
    return 1;
  }
  fclose(o);
  rfm_scan_destroy(s);
  return 0;
}
