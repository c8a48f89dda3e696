"""TEST INFRASTRUCTURE -- the "nco" mixer of one station of a wideband capture, composed like oracle/wideband.py's
OracleStation:

    u8 -> float (RTL_SDR_Source.cpp:207-211), or samples already converted (and corrected) by the caller
    the phase-accumulator NCO at -f_k (oracle/nco.py); its phase runs on across front-end blocks and calls
    CRDSDownConvert::SetWfmDataRate(Fs, bw) at 0 Hz + ProcessData per front-end block
    cFmDecoder(out_rate, 0, 48000, 15000, 1)::ProcessStream per `blocks_per_call` blocks

Only tests/ and bench scripts may import this.
"""
from __future__ import annotations

import numpy as np

from . import nco, port
from .wideband import OracleStation, _P


class OracleNcoStation(OracleStation):
    def __init__(self, f_station: float, fs: float = 50.0e6, front_block: int = 32000, blocks_per_call: int = 64,
                 max_bw: float = 100000.0):
        # any mixer other than "osc" leaves the down-converter at 0 Hz; no shifter is made for "nco"
        super().__init__(f_station, fs, front_block, blocks_per_call, mixer="nco", max_bw=max_bw)
        self.nco = nco.Nco(-f_station, np.float32(fs))

    def baseband(self, capture_u8: np.ndarray) -> np.ndarray:
        """capture [blocks * front_block, 2] u8 -> decimated complex baseband [m, 2]."""
        return self.baseband_cf32(port.u8_to_cf32(capture_u8))

    def baseband_cf32(self, x: np.ndarray) -> np.ndarray:
        """converted (and corrected) float samples [blocks * front_block, 2] -> decimated complex baseband [m, 2]."""
        out = []
        for b in range(x.shape[0] // self.front_block):
            z = np.ascontiguousarray(self.nco.mix(x[b * self.front_block:(b + 1) * self.front_block]))
            y = np.zeros_like(z)
            k = self.L.rfo_rdsdc_process(self.dc, z.shape[0], _P(z), _P(y))
            out.append(y[:k].copy())
        return np.concatenate(out)
