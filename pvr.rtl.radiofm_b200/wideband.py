"""Wideband front end (SURVEY.md section 8d C5 / 8f N3): S stations of ONE shared capture, each mixed to baseband,
decimated by CRDSDownConvert's SetWfmDataRate chain (7 x HB51 at 50 MS/s -> 390 625 S/s) and demodulated by a
cFmDecoder(390625, 0, 48000, 15000, downsample = 1) -- all on the device, composed from the C-ABI primitives through
device pointers.  Host logic only; the arithmetic lives in libradiofm_b200.so.

Two mixers, both reference classes:
  "osc"       CRDSDownConvert::SetFrequency(-f_k): the NCO_OSC rotating vector inside ProcessData (DownConvert.cpp:438-442).
              Bit-exact needs the sequential float recurrence, one lane per station: latency-bound (~60 cycles / sample),
              independent of the station count.
  "freqshift" cFreqShift(-f_k, Fs) with Reset() before every phase-coherent front-end block (f_k * L / Fs integer), then
              CRDSDownConvert at 0 Hz (whose oscillator settles into a 4-cycle).  Fully parallel; the reference's float32
              phase costs it SNR (SURVEY.md section 0.8), parity is against the reference all the same.  Because the
              shifter restarts every block its (cos, sin) sequence is a per-station table of L entries, made once by
              running rfm_freqshift on a block of ones and handed to the down-converter (rfm_downconvert_set_premix):
              one fused kernel per call, nothing intermediate in HBM.
  "freqshift_unfused"  the same arithmetic as separate primitive calls (64 x rfm_freqshift + one rfm_downconvert over
              an S x 2 M complex buffer); kept as a cross-check of the primitives' device entry points.
And one mixer the project defines itself (DESIGN.md section 15):
  "nco"       the phase-accumulator NCO (rfm_downconvert_set_nco(-f_k)) in front of CRDSDownConvert at 0 Hz: a 32-bit
              phase per sample from its index, a phasor from three 256-entry tables (about -133 dBc).  Any frequency
              within +-fs / 2, no phase-coherence condition, the phase continuous across calls, and the cost of the
              freqshift table.

The capture is u8 (RTL-SDR) by default; input_format = "s8" (HackRF), "s16" (the SoapySDR / UHD host format) or "cf32"
takes the other rfm_iq_format formats, converted inside the first kernel that reads the capture.  iq_correction (an
IqCorrection, e.g. from estimate_iq_correction) removes a zero-IF receiver's DC offset and IQ imbalance in that same
kernel, right after the conversion.
"""
from __future__ import annotations

import numpy as np

from . import DownConvertBatch, FmDecoderBatch, FreqShiftBatch, iq_format, iq_format_bytes


class WidebandReceiver:
    def __init__(self, torch, station_freqs, fs: float = 50.0e6, front_block: int = 32000, blocks_per_call: int = 64,
                 mixer: str = "osc", max_bw: float = 100000.0, device: int = 0, lanes_sms: int = 8, n_slots: int = 3,
                 input_format="u8", iq_correction=None):
        if mixer not in ("osc", "freqshift", "freqshift_unfused", "nco"):
            raise ValueError(f"unknown mixer {mixer!r}: use \"osc\", \"freqshift\", \"freqshift_unfused\" or \"nco\"")
        self.torch, self.mixer, self.fs = torch, mixer, fs
        self._fmt = iq_format(input_format)
        self._esz = iq_format_bytes(self._fmt)
        self.freqs = np.ascontiguousarray(station_freqs, dtype=np.float64)
        self.S = S = self.freqs.size
        self.front_block, self.blocks_per_call = front_block, blocks_per_call
        self.n_call = front_block * blocks_per_call
        dev = torch.device("cuda", device)
        if mixer in ("osc", "nco"):
            self.shift = None
            self.dc = DownConvertBatch(-self.freqs if mixer == "osc" else np.zeros(S), fs, max_bw, wfm=True,
                                       max_len=self.n_call, device=device)
            if mixer == "nco":
                self.dc.set_nco(-self.freqs)
        else:
            for f in self.freqs:
                assert abs(f * front_block / fs - round(f * front_block / fs)) < 1e-9, "blocks must be phase-coherent"
            self.shift = FreqShiftBatch(-self.freqs, fs, max_len=front_block, device=device)
            self.dc = DownConvertBatch(np.zeros(S), fs, max_bw, wfm=True, max_len=self.n_call, device=device)
            if mixer == "freqshift":
                ones = np.zeros((S, front_block, 2), dtype=np.float32)
                ones[:, :, 0] = 1.0
                self.table = torch.from_numpy(self.shift.process_cf32(ones)).to(dev)   # [S][L] (cos, sin) after Reset()
                self.dc.set_premix(self.table.data_ptr(), front_block, front_block)
            else:
                self.mixed = torch.empty((S, self.n_call, 2), dtype=torch.float32, device=dev)
        # the correction goes to whichever object reads the capture: the shifter in the unfused form (the down-converter
        # then reads mixed cf32 rows), the down-converter otherwise (the shifter only made the pre-mix table)
        if iq_correction is not None:
            (self.shift if mixer == "freqshift_unfused" else self.dc).set_iq_correction(iq_correction)
        self.n_bb = self.n_call >> self.dc.n_stages
        # The demodulator's lanes kernel (one warp per 32 stations, a latency chain) gets an SM partition of its own and
        # the front end runs on the demodulator's companion stream, i.e. on the OTHER SMs: sharing SMs with the
        # decimation chain's CTAs stretched the lanes kernel from 2.5 to 3.3 ms per call at 100 stations
        self.dec = FmDecoderBatch(self.dc.output_rate, 0.0, downsample=1, n_streams=S, max_block_len=self.n_bb,
                                  device=device, lanes_sms=lanes_sms if lanes_sms >= 8 else 1)
        self.audio_stride = max(self.dec.max_audio_floats(self.n_bb), 2)
        # three slots: the front end of call k+1 runs while the demodulator (latency-bound lanes) still works on call k.
        # With two, the front end of k+1 had to wait for the END of call k-1 and the step was (front end + demodulator
        # entry + lanes + audio tail) / 2 = 3.0 ms at 100 stations; with three it is the lanes kernel's own chain
        self.n_slots = n_slots
        self.bbs = [torch.empty((S, self.n_bb, 2), dtype=torch.float32, device=dev) for _ in range(self.n_slots)]
        self.audios = [torch.empty((S, self.audio_stride), dtype=torch.float32, device=dev) for _ in range(self.n_slots)]
        # the front end and the demodulator are submitted on different streams: on one stream the front end of call k+1
        # would queue behind the demodulator's entry kernels of call k and the step would be their SUM (3.1 ms measured at
        # 100 stations) instead of the longer of the two (the lanes kernel, 2.5 ms)
        self.s_front = torch.cuda.ExternalStream(self.dec.companion_stream(), device=dev)
        self.s_dec = torch.cuda.Stream(device=dev)
        self.s_done = torch.cuda.Stream(device=dev)
        self.ev = [None] * self.n_slots
        self.calls = 0
        self.bb, self.audio = self.bbs[0], self.audios[0]

    def close(self):
        for o in (self.shift, self.dc, self.dec):
            if o is not None:
                o.close()

    def process_device(self, d_capture_ptr: int) -> int:
        """One call = blocks_per_call front-end blocks of the shared capture ([n_call] samples of the input format at
        d_capture_ptr, aligned to the sample size, ready on the
        current stream).  Only enqueues; returns the audio floats per station that self.audio (this call's slot) will hold
        once wait() has ordered the current stream after the call."""
        torch = self.torch
        slot = self.calls % self.n_slots
        sf = self.s_front.cuda_stream
        self.s_front.wait_stream(torch.cuda.current_stream())
        if self.ev[slot] is not None:
            self.s_front.wait_event(self.ev[slot])            # the slot's previous call has left the demodulator
        bb, audio = self.bbs[slot], self.audios[slot]
        if self.mixer in ("osc", "freqshift", "nco"):
            m = self.dc.process_iq_device(self._fmt, True, d_capture_ptr, self.n_call, bb.data_ptr(), self.n_bb,
                                          self.n_call, sf)
        else:
            for b in range(self.blocks_per_call):
                self.shift.reset()
                self.shift.process_iq_device(self._fmt, True, d_capture_ptr + self._esz * b * self.front_block,
                                             self.front_block, self.mixed.data_ptr() + 8 * b * self.front_block,
                                             self.n_call, self.front_block)
            self.s_front.wait_stream(torch.cuda.default_stream())
            m = self.dc.process_device(0, self.mixed.data_ptr(), self.n_call, bb.data_ptr(), self.n_bb, self.n_call, sf)
        assert m == self.n_bb
        ev_bb = torch.cuda.Event()
        ev_bb.record(self.s_front)
        self.s_dec.wait_event(ev_bb)
        k = self.dec.process_cf32_device(bb.data_ptr(), self.n_bb, self.n_bb, audio.data_ptr(), self.audio_stride,
                                         self.s_dec.cuda_stream)
        self.dec.wait(self.s_done.cuda_stream)
        self.ev[slot] = torch.cuda.Event()
        self.ev[slot].record(self.s_done)
        if self.mixer == "freqshift_unfused":
            torch.cuda.default_stream().wait_event(self.ev[slot])   # self.mixed is single-buffered
        self.calls += 1
        self.bb, self.audio = bb, audio
        return k

    def wait(self):
        """Order the current stream after every call enqueued so far."""
        for e in self.ev:
            if e is not None:
                self.torch.cuda.current_stream().wait_event(e)

    def process_u8(self, capture_u8: np.ndarray) -> np.ndarray:
        """Host convenience: capture [n_call, 2] uint8 -> audio [S, floats]."""
        torch = self.torch
        cap = torch.from_numpy(np.ascontiguousarray(capture_u8, dtype=np.uint8).reshape(self.n_call, 2)).to(self.bb.device)
        k = self.process_device(cap.data_ptr())
        self.wait()
        torch.cuda.synchronize()
        return self.audio[:, :k].cpu().numpy()

    def process_iq(self, capture: np.ndarray) -> np.ndarray:
        """Host convenience: capture [n_call, 2] of the input format's dtype (uint8 / int8 / int16 / float32, or
        [n_call] complex64 for cf32) -> audio [S, floats]."""
        torch = self.torch
        a = np.asarray(capture)
        if a.dtype == np.complex64:
            a = np.ascontiguousarray(a).view(np.float32)
        if iq_format(a.dtype) != self._fmt:
            raise ValueError(f"capture dtype {a.dtype} is not the receiver's input format")
        cap = torch.from_numpy(np.ascontiguousarray(a).reshape(self.n_call, 2)).to(self.bb.device)
        k = self.process_device(cap.data_ptr())
        self.wait()
        torch.cuda.synchronize()
        return self.audio[:, :k].cpu().numpy()
