"""radiofm_b200 -- Python binding (ctypes) of the C ABI in include/radiofm_b200.h.

The product is the shared library ``libradiofm_b200.so`` (hand-written sm_100a CUDA kernels + C++
host); this module only loads it and wraps the calls for tests/ and bench.py.  There is no Python or
CPU implementation of the chain behind it: if the library or a B200 is missing, creation fails loudly.

The directory is called ``pvr.rtl.radiofm_b200`` (not importable by dotted name); load it with
``importlib`` under the module name ``radiofm_b200`` -- see ``load_package()`` in tests/conftest.py or
__graft_entry__.py.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RFM_LIB_PATH") or os.path.join(_HERE, "libradiofm_b200.so")  # override: tuning experiments

RFM_OK = 0
_u8p = C.POINTER(C.c_uint8)
_u16p = C.POINTER(C.c_uint16)
_u32p = C.POINTER(C.c_uint32)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)


class RfmConfig(C.Structure):
    _fields_ = [("sample_rate_if", C.c_double), ("tuning_offset", C.c_double), ("sample_rate_pcm", C.c_double),
                ("bandwidth_pcm", C.c_double), ("downsample", C.c_uint32), ("us_deemphasis", C.c_int32),
                ("n_streams", C.c_uint32), ("max_block_len", C.c_uint32), ("device", C.c_int32),
                ("n_groups", C.c_uint32), ("lanes_sms", C.c_uint32), ("fir_fused", C.c_uint32)]


class RfmStreamStatus(C.Structure):
    _fields_ = [("stereo_detected", C.c_int32), ("interface_level", C.c_float), ("baseband_level", C.c_float),
                ("baseband_mean", C.c_float), ("pilot_level", C.c_float), ("tuning_offset", C.c_float)]


EXPORTED_SYMBOLS = (
    "rfm_last_error", "rfm_version", "rfm_launch_count", "rfm_config_default", "rfm_decoder_create",
    "rfm_decoder_destroy", "rfm_decoder_reset", "rfm_decoder_max_audio_floats", "rfm_decoder_process_u8",
    "rfm_decoder_process_cf32", "rfm_decoder_submit_u8", "rfm_decoder_process_u8_device", "rfm_decoder_process_cf32_device", "rfm_decoder_wait",
    "rfm_decoder_synchronize", "rfm_decoder_demod_repairs",
    "rfm_decoder_rds_take_groups", "rfm_decoder_rds_take_bits", "rfm_decoder_rds_take_uecp", "rfm_decoder_get_status",
    "rfm_rdsgroup_create", "rfm_rdsgroup_destroy", "rfm_rdsgroup_reset", "rfm_rdsgroup_decode", "rfm_rdsgroup_take_uecp",
    "rfm_rdsgroup_channel_name", "rfm_uecp_stuff_frame",
    "rfm_demux_create", "rfm_demux_destroy", "rfm_demux_decoder", "rfm_demux_write_u8", "rfm_demux_end",
    "rfm_demux_queued_samples", "rfm_demux_set_stream_change", "rfm_demux_read", "rfm_demux_audio_level",
    "rfm_demux_signal_status", "rfm_source_block_length", "rfm_demux_set_source_block_length", "rfm_demux_source_cb",
    "rfm_demux_short_reads",
    "rfm_rtlsdr_device_count", "rfm_rtlsdr_open", "rfm_rtlsdr_configure", "rfm_rtlsdr_close", "rfm_rtlsdr_get_sample_rate",
    "rfm_rtlsdr_get_frequency", "rfm_rtlsdr_set_frequency", "rfm_rtlsdr_get_tuner_gain", "rfm_rtlsdr_block_length",
    "rfm_rtlsdr_restarts", "rfm_rtlsdr_error",
    "rfm_decoder_constants", "rfm_decoder_table", "rfm_plan_constants", "rfm_plan_table", "rfm_decoder_set_profiling",
    "rfm_decoder_companion_stream",
    "rfm_decoder_profile_read", "rfm_decoder_tap", "rfm_rdssync_create",
    "rfm_rdssync_destroy", "rfm_rdssync_reset", "rfm_rdssync_push_bits", "rfm_rdssync_take_groups",
    "rfm_rds_check_block", "rfm_math_probe", "rfm_div_selftest", "rfm_freqshift_create",
    "rfm_freqshift_destroy", "rfm_freqshift_reset", "rfm_freqshift_process_cf32", "rfm_freqshift_process_u8",
    "rfm_freqshift_process_device", "rfm_downconvert_create", "rfm_downconvert_destroy", "rfm_downconvert_output_rate",
    "rfm_downconvert_stages", "rfm_downconvert_set_frequency", "rfm_downconvert_reset", "rfm_downconvert_process_cf32",
    "rfm_downconvert_process_u8", "rfm_downconvert_process_device", "rfm_downconvert_set_premix",
    "rfm_iir_create", "rfm_iir_destroy", "rfm_iir_init", "rfm_iir_coefficients", "rfm_iir_process_real",
    "rfm_iir_process_complex", "rfm_iir_process_two", "rfm_iir_process_device",
    "rfm_fir_create", "rfm_fir_destroy", "rfm_fir_init_lp", "rfm_fir_init_hp", "rfm_fir_design", "rfm_fir_init_const", "rfm_fir_taps", "rfm_fir_process_real",
    "rfm_fir_process_complex", "rfm_fir_process_two", "rfm_fir_process_device",
    "rfm_downsample_create", "rfm_downsample_destroy", "rfm_downsample_reset", "rfm_downsample_coefficients",
    "rfm_downsample_max_outputs", "rfm_downsample_process_complex", "rfm_downsample_process_real",
    "rfm_downsample_process_complex_device", "rfm_downsample_process_real_device",
    "rfm_rdsproc_create", "rfm_rdsproc_destroy", "rfm_rdsproc_process_rate", "rfm_rdsproc_reset", "rfm_rdsproc_process",
    "rfm_rdsproc_process_device", "rfm_rdsproc_take_bits", "rfm_rdsproc_take_groups",
    "rfm_scan_config_default", "rfm_scan_create", "rfm_scan_destroy", "rfm_scan_run_u8", "rfm_scan_spectrum",
    "rfm_scan_channel_power", "rfm_scan_stations", "rfm_scan_timing",
    "rfm_iq_format_bytes", "rfm_decoder_process_iq", "rfm_decoder_submit_iq", "rfm_decoder_process_iq_device",
    "rfm_freqshift_process_iq", "rfm_freqshift_process_iq_device", "rfm_downconvert_process_iq",
    "rfm_downconvert_process_iq_device", "rfm_scan_run",
    "rfm_iq_estimate", "rfm_downconvert_set_iq_correction", "rfm_freqshift_set_iq_correction",
    "rfm_scan_set_iq_correction", "rfm_scan_iq_correction",
    "rfm_downconvert_set_nco", "rfm_scan_set_mixer",
)

# rfm_iq_format (include/radiofm_b200.h): interleaved I,Q; s8 = v * 2^-7, s16 = v * 2^-15 (exact), full scale of the container
IQ_U8, IQ_S8, IQ_S16, IQ_CF32 = 0, 1, 2, 3
_IQ_NAMES = {"u8": IQ_U8, "uint8": IQ_U8, "s8": IQ_S8, "int8": IQ_S8, "s16": IQ_S16, "int16": IQ_S16,
             "cf32": IQ_CF32, "float32": IQ_CF32, "complex64": IQ_CF32}


def iq_format(f) -> int:
    """IQ format of a dtype (numpy or torch: uint8, int8, int16, float32 / complex64), a name ("u8", "s8", "s16",
    "cf32") or an rfm_iq_format value."""
    if isinstance(f, (int, np.integer)) and not isinstance(f, bool):
        if int(f) not in (IQ_U8, IQ_S8, IQ_S16, IQ_CF32):
            raise ValueError(f"unknown IQ format {f}")
        return int(f)
    name = str(f).replace("torch.", "")
    if name not in _IQ_NAMES:
        try:
            name = str(np.dtype(f))
        except TypeError:
            pass
    if name not in _IQ_NAMES:
        raise ValueError(f"no IQ format for {f!r}: use uint8, int8, int16 or float32 / complex64")
    return _IQ_NAMES[name]


def iq_format_bytes(f) -> int:
    """Bytes per complex sample of an IQ format: 2, 2, 4, 8."""
    return int(lib().rfm_iq_format_bytes(iq_format(f)))


_IQ_DTYPES = {IQ_U8: np.uint8, IQ_S8: np.int8, IQ_S16: np.int16, IQ_CF32: np.float32}


def _iq_host(iq, rows: int | None = None):
    """Host IQ -> (format, C-contiguous array with a trailing (I, Q) axis); rows: reshape to [rows, n, 2]."""
    a = np.asarray(iq)
    if a.dtype == np.complex64:
        a = np.ascontiguousarray(a).view(np.float32)
    fmt = iq_format(a.dtype)
    a = np.ascontiguousarray(a, dtype=_IQ_DTYPES[fmt])
    return fmt, (a.reshape(rows, -1, 2) if rows else a.reshape(-1, 2))


class RfmIqCorrection(C.Structure):
    """rfm_iq_correction (include/radiofm_b200.h)."""
    _fields_ = [("dc_i", C.c_float), ("dc_q", C.c_float), ("a", C.c_float), ("b", C.c_float),
                ("imbalance_valid", C.c_int32)]


@dataclasses.dataclass(frozen=True)
class IqCorrection:
    """Frequency-flat IQ correction of a capture (rfm_iq_correction): y = (I - dc_i) + j (a (Q - dc_q) + b (I - dc_i)),
    in float32 after the format conversion.  imbalance_valid False: a = 1, b = 0 were forced (degenerate statistics)."""
    dc_i: np.float32
    dc_q: np.float32
    a: np.float32 = np.float32(1.0)
    b: np.float32 = np.float32(0.0)
    imbalance_valid: bool = True

    def _c(self) -> RfmIqCorrection:
        return RfmIqCorrection(float(np.float32(self.dc_i)), float(np.float32(self.dc_q)), float(np.float32(self.a)),
                               float(np.float32(self.b)), int(bool(self.imbalance_valid)))

    @staticmethod
    def _from_c(c: RfmIqCorrection) -> "IqCorrection":
        return IqCorrection(np.float32(c.dc_i), np.float32(c.dc_q), np.float32(c.a), np.float32(c.b),
                            bool(c.imbalance_valid))


def _corr_arg(c):
    if c is None:
        return None
    if not isinstance(c, IqCorrection):
        raise TypeError(f"expected an IqCorrection or None, got {type(c).__name__}")
    return C.byref(c._c())


def estimate_iq_correction(capture, fmt=None, n: int | None = None, device: int = -1) -> IqCorrection:
    """rfm_iq_estimate: the blind DC / gain / phase estimate of one capture.  capture: a host array [n, 2] of uint8 /
    int8 / int16 / float32 ([n] complex64), a contiguous CUDA tensor of those dtypes (complete before the call), or a
    device pointer (int) with its format and sample count."""
    out = RfmIqCorrection()
    if isinstance(capture, (int, np.integer)):
        if fmt is None or n is None:
            raise ValueError("a device pointer needs fmt and n")
        _check(lib().rfm_iq_estimate(iq_format(fmt), C.c_void_p(int(capture)), int(n), 1, device, C.byref(out)))
    elif hasattr(capture, "data_ptr") and getattr(capture, "is_cuda", False):
        f = iq_format(capture.dtype)
        if not capture.is_contiguous():
            raise ValueError("device capture must be contiguous")
        cnt = capture.numel() // (1 if f == IQ_CF32 and capture.is_complex() else 2)
        dev = capture.device.index if device < 0 and capture.device.index is not None else device
        _check(lib().rfm_iq_estimate(f, C.c_void_p(capture.data_ptr()), cnt, 1, dev, C.byref(out)))
    else:
        f, cap = _iq_host(capture)
        _check(lib().rfm_iq_estimate(f, cap.ctypes.data_as(C.c_void_p), cap.shape[0], 0, device, C.byref(out)))
    return IqCorrection._from_c(out)


_ADD_FRAME_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_uint32)
_SET_NAME_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_char_p)
_SETTING_CB = C.CFUNCTYPE(C.c_int, C.c_void_p)


class ScanConfig(C.Structure):
    """rfm_scan_config (include/radiofm_b200.h)."""
    _fields_ = [("sample_rate", C.c_double), ("raster_first", C.c_double), ("raster_step", C.c_double),
                ("raster_count", C.c_uint32), ("min_snr_db", C.c_double), ("device", C.c_int32)]


class ScanStation(C.Structure):
    """rfm_scan_station (include/radiofm_b200.h)."""
    _fields_ = [("freq", C.c_double), ("power_dbfs", C.c_float), ("snr_db", C.c_float),
                ("stereo_detected", C.c_int32), ("pilot_level", C.c_float), ("interface_level", C.c_float),
                ("baseband_level", C.c_float), ("rds_groups", C.c_uint32), ("pi", C.c_int32), ("ps", C.c_char * 9)]


class RdsGroupCallbacks(C.Structure):
    """rfm_rdsgroup_callbacks (include/radiofm_b200.h)."""
    _fields_ = [("user", C.c_void_p), ("add_uecp_frame", _ADD_FRAME_CB), ("set_channel_name", _SET_NAME_CB),
                ("is_setting_active", _SETTING_CB)]


class DemuxPacket(C.Structure):
    """rfm_demux_packet (include/radiofm_b200.h)."""
    _fields_ = [("stream_id", C.c_int32), ("size_bytes", C.c_uint32), ("pts", C.c_double), ("duration", C.c_double),
                ("data", C.c_void_p)]


DEMUX_STREAMCHANGE = -11
DEMUX_END = 1


class RadioFmError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a into the in-tree libradiofm_b200.so (nvcc cross-compiles)."""
    out = subprocess.run(["sh", os.path.join(_HERE, "csrc", "build.sh")], capture_output=True, text=True)
    if out.returncode != 0:
        raise RadioFmError("build failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RadioFmError(f"{LIB_PATH} is missing: run __graft_entry__.build() (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        L.rfm_last_error.restype = C.c_char_p
        L.rfm_version.restype = C.c_char_p
        L.rfm_launch_count.restype = C.c_uint64
        L.rfm_config_default.argtypes = [C.POINTER(RfmConfig)]
        L.rfm_decoder_create.argtypes = [C.POINTER(RfmConfig), C.POINTER(C.c_void_p)]
        L.rfm_decoder_destroy.argtypes = [C.c_void_p]
        L.rfm_decoder_reset.argtypes = [C.c_void_p]
        L.rfm_decoder_max_audio_floats.restype = C.c_uint32
        L.rfm_decoder_max_audio_floats.argtypes = [C.c_void_p, C.c_uint32]
        L.rfm_decoder_process_u8.argtypes = [C.c_void_p, _u8p, C.c_uint32, _f32p, C.c_size_t, _u32p]
        L.rfm_decoder_submit_u8.argtypes = [C.c_void_p, _u8p, C.c_uint32, _f32p, C.c_size_t, _u32p]
        L.rfm_decoder_process_cf32.argtypes = [C.c_void_p, _f32p, C.c_uint32, _f32p, C.c_size_t, _u32p]
        L.rfm_decoder_process_u8_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                                    C.c_size_t, _u32p, C.c_void_p]
        L.rfm_decoder_process_cf32_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                                      C.c_size_t, _u32p, C.c_void_p]
        L.rfm_decoder_wait.argtypes = [C.c_void_p, C.c_void_p]
        L.rfm_decoder_synchronize.argtypes = [C.c_void_p]
        L.rfm_decoder_demod_repairs.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.rfm_decoder_rds_take_groups.argtypes = [C.c_void_p, C.c_uint32, _u16p, C.c_uint32, _u32p]
        L.rfm_decoder_rds_take_uecp.argtypes = [C.c_void_p, C.c_uint32, _u8p, C.c_uint32, _u32p]
        L.rfm_rdsgroup_create.argtypes = [C.POINTER(RdsGroupCallbacks), C.POINTER(C.c_void_p)]
        L.rfm_rdsgroup_destroy.argtypes = [C.c_void_p]
        L.rfm_rdsgroup_reset.argtypes = [C.c_void_p]
        L.rfm_rdsgroup_decode.argtypes = [C.c_void_p, _u16p, C.c_uint32]
        L.rfm_rdsgroup_take_uecp.argtypes = [C.c_void_p, _u8p, C.c_uint32, _u32p]
        L.rfm_rdsgroup_channel_name.argtypes = [C.c_void_p, C.c_char_p]
        L.rfm_demux_create.argtypes = [C.POINTER(RfmConfig), C.POINTER(C.c_void_p)]
        L.rfm_demux_destroy.argtypes = [C.c_void_p]
        L.rfm_demux_decoder.restype = C.c_void_p
        L.rfm_demux_decoder.argtypes = [C.c_void_p]
        L.rfm_demux_write_u8.argtypes = [C.c_void_p, _u8p, C.c_uint32]
        L.rfm_demux_end.argtypes = [C.c_void_p]
        L.rfm_demux_queued_samples.restype = C.c_uint64
        L.rfm_demux_queued_samples.argtypes = [C.c_void_p]
        L.rfm_demux_set_stream_change.argtypes = [C.c_void_p]
        L.rfm_demux_read.argtypes = [C.c_void_p, C.POINTER(DemuxPacket)]
        L.rfm_demux_audio_level.restype = C.c_float
        L.rfm_demux_audio_level.argtypes = [C.c_void_p]
        L.rfm_demux_signal_status.argtypes = [C.c_void_p, _f32p, _f32p, C.POINTER(C.c_int)]
        L.rfm_source_block_length.restype = C.c_uint32
        L.rfm_source_block_length.argtypes = [C.c_uint32]
        L.rfm_demux_set_source_block_length.argtypes = [C.c_void_p, C.c_uint32]
        L.rfm_demux_source_cb.restype = None
        L.rfm_demux_source_cb.argtypes = [_u8p, C.c_uint32, C.c_void_p]
        L.rfm_demux_short_reads.restype = C.c_uint64
        L.rfm_demux_short_reads.argtypes = [C.c_void_p]
        L.rfm_uecp_stuff_frame.restype = C.c_uint32
        L.rfm_uecp_stuff_frame.argtypes = [_u8p, C.c_uint32, _u8p, C.c_uint32]
        L.rfm_decoder_rds_take_bits.argtypes = [C.c_void_p, C.c_uint32, _u8p, C.c_uint32, _u32p]
        L.rfm_decoder_get_status.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(RfmStreamStatus)]
        L.rfm_decoder_constants.argtypes = [C.c_void_p, _f64p, C.c_uint32]
        L.rfm_decoder_table.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_uint32, _u32p]
        L.rfm_plan_constants.argtypes = [C.POINTER(RfmConfig), _f64p, C.c_uint32]
        L.rfm_plan_table.argtypes = [C.POINTER(RfmConfig), C.c_int, _f32p, C.c_uint32, _u32p]
        L.rfm_decoder_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.rfm_decoder_companion_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.rfm_decoder_profile_read.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p, C.c_uint32, _f64p,
                                               C.POINTER(C.c_uint64)]
        L.rfm_decoder_tap.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, _f32p, C.c_uint32, _u32p]
        L.rfm_rdssync_create.argtypes = [C.POINTER(C.c_void_p)]
        L.rfm_rdssync_destroy.argtypes = [C.c_void_p]
        L.rfm_rdssync_reset.argtypes = [C.c_void_p]
        L.rfm_rdssync_push_bits.argtypes = [C.c_void_p, _u8p, C.c_uint32]
        L.rfm_rdssync_take_groups.argtypes = [C.c_void_p, _u16p, C.c_uint32, _u32p]
        L.rfm_math_probe.argtypes = [C.c_int, _f32p, _f32p, _f32p, C.c_uint32]
        L.rfm_div_selftest.argtypes = [C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.rfm_freqshift_create.argtypes = [C.c_uint32, _f32p, C.c_float, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.rfm_freqshift_destroy.argtypes = [C.c_void_p]
        L.rfm_freqshift_reset.argtypes = [C.c_void_p]
        L.rfm_freqshift_process_cf32.argtypes = [C.c_void_p, _f32p, C.c_uint32]
        L.rfm_freqshift_process_u8.argtypes = [C.c_void_p, _u8p, C.c_int, C.c_uint32, _f32p]
        L.rfm_freqshift_process_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                   C.c_uint32, C.c_void_p]
        L.rfm_downconvert_create.argtypes = [C.c_uint32, _f32p, C.c_float, C.c_float, C.c_int, C.c_uint32, C.c_int,
                                             C.POINTER(C.c_void_p)]
        L.rfm_downconvert_destroy.argtypes = [C.c_void_p]
        L.rfm_downconvert_output_rate.restype = C.c_float
        L.rfm_downconvert_output_rate.argtypes = [C.c_void_p]
        L.rfm_downconvert_stages.restype = C.c_uint32
        L.rfm_downconvert_stages.argtypes = [C.c_void_p, _u32p, C.c_uint32]
        L.rfm_downconvert_set_frequency.argtypes = [C.c_void_p, _f32p]
        L.rfm_downconvert_reset.argtypes = [C.c_void_p]
        L.rfm_downconvert_set_premix.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32]
        L.rfm_downconvert_process_cf32.argtypes = [C.c_void_p, _f32p, C.c_uint32, _f32p, _u32p]
        L.rfm_downconvert_process_u8.argtypes = [C.c_void_p, _u8p, C.c_int, C.c_uint32, _f32p, _u32p]
        L.rfm_downconvert_process_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                     C.c_uint32, _u32p, C.c_void_p]
        for nm in ("iir", "fir"):
            getattr(L, f"rfm_{nm}_create").argtypes = [C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
            getattr(L, f"rfm_{nm}_destroy").argtypes = [C.c_void_p]
            getattr(L, f"rfm_{nm}_process_real").argtypes = [C.c_void_p, _f32p, C.c_uint32]
            getattr(L, f"rfm_{nm}_process_complex").argtypes = [C.c_void_p, _f32p, C.c_uint32]
            getattr(L, f"rfm_{nm}_process_two").argtypes = [C.c_void_p, _f32p, _f32p, C.c_uint32]
            getattr(L, f"rfm_{nm}_process_device").argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                                               C.c_uint32, C.c_void_p]
        L.rfm_iir_init.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float]
        L.rfm_iir_coefficients.argtypes = [C.c_void_p, _f32p]
        L.rfm_fir_init_lp.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _u32p]
        L.rfm_fir_init_hp.argtypes = L.rfm_fir_init_lp.argtypes
        L.rfm_fir_design.argtypes = [C.c_int, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _f32p,
                                     C.c_uint32, _u32p]
        L.rfm_fir_init_const.argtypes = [C.c_void_p, C.c_uint32, _f32p, C.c_float]
        L.rfm_fir_taps.argtypes = [C.c_void_p, _f32p, C.c_uint32, _u32p]
        L.rfm_downsample_create.argtypes = [C.c_uint32, C.c_uint32, C.c_double, C.c_double, C.c_int, C.c_uint32, C.c_int,
                                            C.POINTER(C.c_void_p)]
        L.rfm_downsample_destroy.argtypes = [C.c_void_p]
        L.rfm_downsample_reset.argtypes = [C.c_void_p]
        L.rfm_downsample_coefficients.argtypes = [C.c_void_p, _f32p, C.c_uint32, _u32p]
        L.rfm_downsample_max_outputs.restype = C.c_uint32
        L.rfm_downsample_max_outputs.argtypes = [C.c_void_p, C.c_uint32]
        L.rfm_downsample_process_complex.argtypes = [C.c_void_p, _f32p, _f32p, C.c_uint32, _u32p]
        L.rfm_downsample_process_real.argtypes = [C.c_void_p, _f32p, _f32p, C.c_uint32, _u32p]
        for nm in ("complex", "real"):
            getattr(L, f"rfm_downsample_process_{nm}_device").argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                                                          C.c_size_t, C.c_uint32, _u32p, C.c_void_p]
        L.rfm_rdsproc_create.argtypes = [C.c_uint32, C.c_float, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.rfm_rdsproc_destroy.argtypes = [C.c_void_p]
        L.rfm_rdsproc_process_rate.restype = C.c_float
        L.rfm_rdsproc_process_rate.argtypes = [C.c_void_p]
        L.rfm_rdsproc_reset.argtypes = [C.c_void_p]
        L.rfm_rdsproc_process.argtypes = [C.c_void_p, _f32p, C.c_uint32]
        L.rfm_rdsproc_process_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]
        L.rfm_rdsproc_take_bits.argtypes = [C.c_void_p, C.c_uint32, _u8p, C.c_uint32, _u32p]
        L.rfm_rdsproc_take_groups.argtypes = [C.c_void_p, C.c_uint32, _u16p, C.c_uint32, _u32p]
        L.rfm_scan_config_default.restype = None
        L.rfm_scan_config_default.argtypes = [C.POINTER(ScanConfig)]
        L.rfm_scan_create.argtypes = [C.POINTER(ScanConfig), C.POINTER(C.c_void_p)]
        L.rfm_scan_destroy.restype = None
        L.rfm_scan_destroy.argtypes = [C.c_void_p]
        L.rfm_scan_run_u8.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int]
        L.rfm_scan_spectrum.argtypes = [C.c_void_p, _f32p, C.c_uint32, _u32p]
        L.rfm_scan_channel_power.argtypes = [C.c_void_p, _f64p, C.c_uint32]
        L.rfm_scan_stations.argtypes = [C.c_void_p, C.POINTER(ScanStation), C.c_uint32, _u32p]
        L.rfm_scan_timing.argtypes = [C.c_void_p, _f64p, _f64p]
        L.rfm_iq_format_bytes.restype = C.c_uint32
        L.rfm_iq_format_bytes.argtypes = [C.c_int]
        L.rfm_decoder_process_iq.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, _f32p, C.c_size_t, _u32p]
        L.rfm_decoder_submit_iq.argtypes = L.rfm_decoder_process_iq.argtypes
        L.rfm_decoder_process_iq_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                                    C.c_size_t, _u32p, C.c_void_p]
        L.rfm_freqshift_process_iq.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint32, _f32p]
        L.rfm_freqshift_process_iq_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                                      C.c_size_t, C.c_uint32, C.c_void_p]
        L.rfm_downconvert_process_iq.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint32, _f32p, _u32p]
        L.rfm_downconvert_process_iq_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                                        C.c_size_t, C.c_uint32, _u32p, C.c_void_p]
        L.rfm_scan_run.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_int]
        L.rfm_iq_estimate.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(RfmIqCorrection)]
        L.rfm_downconvert_set_iq_correction.argtypes = [C.c_void_p, C.POINTER(RfmIqCorrection)]
        L.rfm_freqshift_set_iq_correction.argtypes = [C.c_void_p, C.POINTER(RfmIqCorrection)]
        L.rfm_scan_set_iq_correction.argtypes = [C.c_void_p, C.c_int, C.POINTER(RfmIqCorrection)]
        L.rfm_scan_iq_correction.argtypes = [C.c_void_p, C.POINTER(RfmIqCorrection)]
        L.rfm_downconvert_set_nco.argtypes = [C.c_void_p, _f64p]
        L.rfm_scan_set_mixer.argtypes = [C.c_void_p, C.c_int]
        L.rfm_rds_check_block.restype = C.c_uint32
        L.rfm_rds_check_block.argtypes = [C.c_uint32, C.c_uint32, C.c_int, _u32p]
        _lib = L
    return _lib


def _quiet_del(close):
    """__del__ form of a close() method: at interpreter shutdown the module globals may already be gone"""
    def __del__(self):
        try:
            close(self)
        except TypeError:
            pass
    return __del__


def _check(rc: int):
    if rc != RFM_OK:
        raise RadioFmError(f"radiofm_b200 error {rc}: {lib().rfm_last_error().decode()}")


def _p(a, t):
    return a.ctypes.data_as(t)


def launch_count() -> int:
    return int(lib().rfm_launch_count())


_COMPLEX_TAPS = {"demod_in", "rds_dec", "rds_lp"}


def _config(fs_if, tuning_offset, fs_pcm=48000.0, bw_pcm=15000.0, downsample=1, usver=False, n_streams=1,
            max_block_len=65536, device=-1, n_groups=0, lanes_sms=0, fir_fused=0) -> RfmConfig:
    cfg = RfmConfig()
    lib().rfm_config_default(C.byref(cfg))
    cfg.sample_rate_if, cfg.tuning_offset, cfg.sample_rate_pcm, cfg.bandwidth_pcm = fs_if, tuning_offset, fs_pcm, bw_pcm
    cfg.downsample, cfg.us_deemphasis, cfg.n_streams = downsample, int(usver), n_streams
    cfg.max_block_len, cfg.device, cfg.n_groups = max_block_len, device, n_groups
    cfg.lanes_sms = lanes_sms
    cfg.fir_fused = fir_fused
    return cfg


def plan_constants(fs_if, tuning_offset, fs_pcm=48000.0, bw_pcm=15000.0, downsample=1, usver=False) -> np.ndarray:
    """Host-only planner output (no device needed); index list = oracle's rfo_constants / ref_fm_constants."""
    cfg = _config(fs_if, tuning_offset, fs_pcm, bw_pcm, downsample, usver)
    s = np.zeros(64, dtype=np.float64)
    rc = lib().rfm_plan_constants(C.byref(cfg), _p(s, _f64p), 64)
    if rc < 0:
        _check(rc)
    return s


def plan_table(which: int, fs_if, tuning_offset, fs_pcm=48000.0, bw_pcm=15000.0, downsample=1, usver=False) -> np.ndarray:
    cfg = _config(fs_if, tuning_offset, fs_pcm, bw_pcm, downsample, usver)
    out = np.zeros(4096, dtype=np.float32)
    k = C.c_uint32(0)
    _check(lib().rfm_plan_table(C.byref(cfg), which, _p(out, _f32p), out.size, C.byref(k)))
    return out[:k.value].copy()


class FmDecoderBatch:
    """n_streams x cFmDecoder (FmDecode.h:99-165) on one B200."""

    def __init__(self, fs_if: float, tuning_offset: float, fs_pcm: float = 48000.0, bw_pcm: float = 15000.0,
                 downsample: int = 1, usver: bool = False, n_streams: int = 1, max_block_len: int = 65536,
                 device: int = -1, n_groups: int = 0, lanes_sms: int = 0, fir_fused: int = 0):
        cfg = _config(fs_if, tuning_offset, fs_pcm, bw_pcm, downsample, usver, n_streams, max_block_len, device,
                      n_groups, lanes_sms, fir_fused)
        self.n_streams = n_streams
        self._h = C.c_void_p()
        _check(lib().rfm_decoder_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_decoder_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        _check(lib().rfm_decoder_reset(self._h))

    def max_audio_floats(self, n: int) -> int:
        return int(lib().rfm_decoder_max_audio_floats(self._h, n))

    # ---- host buffers (numpy) ----
    def process_u8(self, iq_u8: np.ndarray) -> np.ndarray:
        """iq_u8 [S, n, 2] uint8 -> audio [S, floats] float32 (interleaved L,R)."""
        iq_u8 = np.ascontiguousarray(iq_u8, dtype=np.uint8).reshape(self.n_streams, -1, 2)
        n = iq_u8.shape[1]
        stride = max(self.max_audio_floats(n), 2)
        audio = np.empty((self.n_streams, stride), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_process_u8(self._h, _p(iq_u8, _u8p), n, _p(audio, _f32p), stride, C.byref(k)))
        return audio[:, :k.value].copy()

    def process_cf32(self, iq: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.float32).reshape(self.n_streams, -1, 2)
        n = iq.shape[1]
        stride = max(self.max_audio_floats(n), 2)
        audio = np.empty((self.n_streams, stride), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_process_cf32(self._h, _p(iq, _f32p), n, _p(audio, _f32p), stride, C.byref(k)))
        return audio[:, :k.value].copy()

    def process_iq(self, iq: np.ndarray, submit: bool = False) -> np.ndarray:
        """iq [S, n, 2] of uint8 / int8 / int16 / float32 (or [S, n] complex64) -> audio [S, floats] float32.  The
        format comes from the dtype (iq_format).  submit: enqueue only (rfm_decoder_submit_iq); the audio is valid after
        synchronize(), and iq must stay alive until then."""
        fmt, iq = _iq_host(iq, self.n_streams)
        n = iq.shape[1]
        stride = max(self.max_audio_floats(n), 2)
        audio = np.empty((self.n_streams, stride), dtype=np.float32)
        k = C.c_uint32(0)
        call = lib().rfm_decoder_submit_iq if submit else lib().rfm_decoder_process_iq
        _check(call(self._h, fmt, iq.ctypes.data_as(C.c_void_p), n, _p(audio, _f32p), stride, C.byref(k)))
        if submit:
            self._submitted = (iq, audio)
            return audio[:, :k.value]
        return audio[:, :k.value].copy()

    # ---- device buffers (raw pointers, e.g. torch tensors' data_ptr()) ----
    def process_iq_device(self, fmt, d_iq_ptr: int, iq_stride: int, n: int, d_audio_ptr: int, audio_stride: int,
                          cuda_stream: int = 0) -> int:
        """fmt: iq_format() of the device rows (a dtype such as torch.int16, a name or an rfm_iq_format value)."""
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_process_iq_device(self._h, iq_format(fmt), C.c_void_p(d_iq_ptr), iq_stride, n,
                                                   C.c_void_p(d_audio_ptr), audio_stride, C.byref(k),
                                                   C.c_void_p(cuda_stream)))
        return int(k.value)

    def process_u8_device(self, d_iq_ptr: int, iq_stride: int, n: int, d_audio_ptr: int, audio_stride: int,
                          cuda_stream: int = 0) -> int:
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_process_u8_device(self._h, C.c_void_p(d_iq_ptr), iq_stride, n,
                                                   C.c_void_p(d_audio_ptr), audio_stride, C.byref(k),
                                                   C.c_void_p(cuda_stream)))
        return int(k.value)

    def process_cf32_device(self, d_iq_ptr: int, iq_stride: int, n: int, d_audio_ptr: int, audio_stride: int,
                            cuda_stream: int = 0) -> int:
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_process_cf32_device(self._h, C.c_void_p(d_iq_ptr), iq_stride, n,
                                                     C.c_void_p(d_audio_ptr), audio_stride, C.byref(k),
                                                     C.c_void_p(cuda_stream)))
        return int(k.value)

    def wait(self, cuda_stream: int = 0):
        """Order `cuda_stream` after every block enqueued so far (device entry points only enqueue)."""
        _check(lib().rfm_decoder_wait(self._h, C.c_void_p(cuda_stream)))

    def demod_repairs(self) -> int:
        v = C.c_uint64(0)
        _check(lib().rfm_decoder_demod_repairs(self._h, C.byref(v)))
        return int(v.value)

    def synchronize(self):
        _check(lib().rfm_decoder_synchronize(self._h))

    # ---- RDS / telemetry ----
    def take_uecp(self, stream: int = 0, cap: int = 1 << 16) -> bytes:
        """UECP byte stream of the stream's group decoder (cRDSGroupDecoder + AddUECPDataFrame framing)."""
        out = np.zeros(cap, dtype=np.uint8)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_rds_take_uecp(self._h, stream, _p(out, _u8p), cap, C.byref(k)))
        return out[:k.value].tobytes()

    def take_groups(self, stream: int = 0, max_groups: int = 4096) -> np.ndarray:
        out = np.zeros((max_groups, 4), dtype=np.uint16)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_rds_take_groups(self._h, stream, _p(out, _u16p), max_groups, C.byref(k)))
        return out[:k.value].copy()

    def take_bits(self, stream: int = 0, max_bits: int = 1 << 20) -> np.ndarray:
        out = np.zeros(max_bits, dtype=np.uint8)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_rds_take_bits(self._h, stream, _p(out, _u8p), max_bits, C.byref(k)))
        return out[:k.value].copy()

    def status(self, stream: int = 0) -> dict:
        s = RfmStreamStatus()
        _check(lib().rfm_decoder_get_status(self._h, stream, C.byref(s)))
        return {"stereo": bool(s.stereo_detected), "if_level": np.float32(s.interface_level),
                "bb_level": np.float32(s.baseband_level), "bb_mean": np.float32(s.baseband_mean),
                "pilot_level": np.float32(s.pilot_level), "tuning_offset": np.float32(s.tuning_offset)}

    def companion_stream(self) -> int:
        """cudaStream_t (as an int) on the FIR side of the decoder's SM partition, for the kernels that make its input."""
        st = C.c_void_p()
        _check(lib().rfm_decoder_companion_stream(self._h, C.byref(st)))
        return int(st.value or 0)

    def set_profiling(self, on: bool):
        _check(lib().rfm_decoder_set_profiling(self._h, int(on)))

    def profile(self) -> dict:
        """{kernel name: (total device ms, launches)} accumulated since set_profiling(True)."""
        out = {}
        name = C.create_string_buffer(64)
        ms, cnt = C.c_double(0), C.c_uint64(0)
        i = 0
        while True:
            rc = lib().rfm_decoder_profile_read(self._h, i, name, 64, C.byref(ms), C.byref(cnt))
            if rc == 1:
                break
            _check(rc)
            out[name.value.decode()] = (ms.value, int(cnt.value))
            i += 1
        return out

    def constants(self) -> np.ndarray:
        s = np.zeros(64, dtype=np.float64)
        rc = lib().rfm_decoder_constants(self._h, _p(s, _f64p), 64)
        if rc < 0:
            _check(rc)
        return s

    def table(self, which: int) -> np.ndarray:
        out = np.zeros(4096, dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_table(self._h, which, _p(out, _f32p), out.size, C.byref(k)))
        return out[:k.value].copy()

    def tap(self, name: str, stream: int = 0) -> np.ndarray:
        out = np.zeros(1 << 18, dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_decoder_tap(self._h, name.encode(), stream, _p(out, _f32p), out.size, C.byref(k)))
        a = out[:k.value].copy()
        return a.reshape(-1, 2) if name in _COMPLEX_TAPS else a


class RdsBlockSync:
    """Host-side RDS block sync / FEC (RDSProcess.cpp:272-431)."""

    def __init__(self):
        self._h = C.c_void_p()
        _check(lib().rfm_rdssync_create(C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_rdssync_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        lib().rfm_rdssync_reset(self._h)

    def push_bits(self, bits: np.ndarray):
        bits = np.ascontiguousarray(bits, dtype=np.uint8)
        _check(lib().rfm_rdssync_push_bits(self._h, _p(bits, _u8p), bits.size))

    def take_groups(self, max_groups: int = 4096) -> np.ndarray:
        out = np.zeros((max_groups, 4), dtype=np.uint16)
        k = C.c_uint32(0)
        _check(lib().rfm_rdssync_take_groups(self._h, _p(out, _u16p), max_groups, C.byref(k)))
        return out[:k.value].copy()


class RdsGroupDecoder:
    """cRDSGroupDecoder (RDSGroupDecoder.cpp:136-1001) on the host: RDS groups -> UECP frames.

    Without callbacks the frames collect in the transport framing of cRadioReceiver::AddUECPDataFrame
    (take_uecp).  With `on_frame(bytes)`, `on_name(bytes) -> bool`, `setting_active() -> bool` they are the three
    calls the reference makes on its cRadioReceiver."""

    def __init__(self, on_frame=None, on_name=None, setting_active=None):
        self._h = C.c_void_p()
        self._cb = RdsGroupCallbacks()
        if on_frame is not None:
            self._cb.add_uecp_frame = _ADD_FRAME_CB(lambda u, f, n: int(bool(on_frame(bytes(f[:n])) or True)))
        if on_name is not None:
            self._cb.set_channel_name = _SET_NAME_CB(lambda u, s: int(bool(on_name(s))))
        if setting_active is not None:
            self._cb.is_setting_active = _SETTING_CB(lambda u: int(bool(setting_active())))
        have = on_frame is not None or on_name is not None or setting_active is not None
        _check(lib().rfm_rdsgroup_create(C.byref(self._cb) if have else None, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_rdsgroup_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        lib().rfm_rdsgroup_reset(self._h)

    def decode(self, groups: np.ndarray):
        g = np.ascontiguousarray(groups, dtype=np.uint16).reshape(-1, 4)
        _check(lib().rfm_rdsgroup_decode(self._h, _p(g, _u16p), g.shape[0]))

    def take_uecp(self, cap: int = 1 << 16) -> bytes:
        out = np.zeros(cap, dtype=np.uint8)
        k = C.c_uint32(0)
        _check(lib().rfm_rdsgroup_take_uecp(self._h, _p(out, _u8p), cap, C.byref(k)))
        return out[:k.value].tobytes()

    def channel_name(self) -> bytes:
        buf = C.create_string_buffer(9)
        _check(lib().rfm_rdsgroup_channel_name(self._h, buf))
        return buf.raw[:8]


class RtlSdrSource:
    """cRtlSdrSource (RTL_SDR_Source.h:21-86) in front of a Demux: librtlsdr bound at run time (rfm_rtlsdr_*)."""
    AUTO_GAIN = -(1 << 31)   # INT_MIN

    def __init__(self, demux: "Demux", library: str | None = None, dev_index: int = 0):
        L = lib()
        L.rfm_rtlsdr_open.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
        L.rfm_rtlsdr_configure.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int]
        L.rfm_rtlsdr_close.argtypes = [C.c_void_p]
        L.rfm_rtlsdr_set_frequency.argtypes = [C.c_void_p, C.c_uint32]
        for n in ("get_sample_rate", "get_frequency", "block_length", "restarts"):
            f = getattr(L, "rfm_rtlsdr_" + n)
            f.argtypes, f.restype = [C.c_void_p], C.c_uint32
        L.rfm_rtlsdr_get_tuner_gain.argtypes = [C.c_void_p]
        L.rfm_rtlsdr_error.argtypes, L.rfm_rtlsdr_error.restype = [C.c_void_p], C.c_char_p
        self._h = C.c_void_p()
        self._demux = demux
        rc = L.rfm_rtlsdr_open(demux._h, library.encode() if library else None, dev_index, C.byref(self._h))
        if rc != RFM_OK:
            raise RadioFmError(f"rfm_rtlsdr_open: error {rc}")

    def configure(self, sample_rate: int, frequency: int, tuner_gain: int = AUTO_GAIN, block_length: int = 65536,
                  agcmode: bool = False):
        rc = lib().rfm_rtlsdr_configure(self._h, sample_rate, frequency, tuner_gain, block_length, int(agcmode))
        if rc != RFM_OK:
            raise RadioFmError(f"rfm_rtlsdr_configure: error {rc}: {lib().rfm_rtlsdr_error(self._h).decode()}")

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_rtlsdr_close(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    sample_rate = property(lambda self: int(lib().rfm_rtlsdr_get_sample_rate(self._h)))
    frequency = property(lambda self: int(lib().rfm_rtlsdr_get_frequency(self._h)))
    tuner_gain = property(lambda self: int(lib().rfm_rtlsdr_get_tuner_gain(self._h)))
    block_length = property(lambda self: int(lib().rfm_rtlsdr_block_length(self._h)))
    restarts = property(lambda self: int(lib().rfm_rtlsdr_restarts(self._h)))

    def set_frequency(self, f: int):
        lib().rfm_rtlsdr_set_frequency(self._h, f)


class Demux:
    """IQ block queue + packetiser of cRadioReceiver (RadioReceiver.cpp:420-542) for one programme."""

    def __init__(self, fs_if, tuning_offset, fs_pcm=48000.0, bw_pcm=15000.0, downsample=1, usver=False,
                 max_block_len=65536, device=-1):
        cfg = _config(fs_if, tuning_offset, fs_pcm, bw_pcm, downsample, usver, 1, max_block_len, device)
        self._h = C.c_void_p()
        _check(lib().rfm_demux_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_demux_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def write_u8(self, iq_u8: np.ndarray):
        iq_u8 = np.ascontiguousarray(iq_u8, dtype=np.uint8).reshape(-1, 2)
        _check(lib().rfm_demux_write_u8(self._h, _p(iq_u8, _u8p), iq_u8.shape[0]))

    def set_source_block_length(self, requested: int):
        _check(lib().rfm_demux_set_source_block_length(self._h, requested))

    def source_cb(self, buf: np.ndarray):
        """what librtlsdr's reader thread would call (cRtlSdrSource::ReadAsyncCB)"""
        buf = np.ascontiguousarray(buf, dtype=np.uint8).reshape(-1)
        lib().rfm_demux_source_cb(_p(buf, _u8p), buf.size, self._h)

    def short_reads(self) -> int:
        return int(lib().rfm_demux_short_reads(self._h))

    def end(self):
        _check(lib().rfm_demux_end(self._h))

    def queued_samples(self) -> int:
        return int(lib().rfm_demux_queued_samples(self._h))

    def set_stream_change(self):
        lib().rfm_demux_set_stream_change(self._h)

    def read(self):
        """-> (stream_id, pts, duration, payload) or None at the end.  payload: float32 array (audio), bytes (UECP)."""
        pkt = DemuxPacket()
        rc = lib().rfm_demux_read(self._h, C.byref(pkt))
        if rc == DEMUX_END:
            return None
        _check(rc)
        if pkt.stream_id == 1:
            n = pkt.size_bytes // 4
            data = np.ctypeslib.as_array(C.cast(pkt.data, _f32p), shape=(n,)).copy() if n else np.zeros(0, np.float32)
        elif pkt.stream_id == 2:
            data = C.string_at(pkt.data, pkt.size_bytes)
        else:
            data = None
        return pkt.stream_id, pkt.pts, pkt.duration, data

    def audio_level(self) -> float:
        return float(lib().rfm_demux_audio_level(self._h))

    def signal_status(self):
        a, b, s = C.c_float(0), C.c_float(0), C.c_int(0)
        _check(lib().rfm_demux_signal_status(self._h, C.byref(a), C.byref(b), C.byref(s)))
        return a.value, b.value, bool(s.value)


def uecp_stuff_frame(frame: bytes) -> bytes:
    """cRadioReceiver::AddUECPDataFrame's framing (RadioReceiver.cpp:387-414)."""
    src = np.frombuffer(frame, dtype=np.uint8)
    out = np.zeros(2 * len(frame) + 2, dtype=np.uint8)
    n = lib().rfm_uecp_stuff_frame(_p(src, _u8p) if len(frame) else None, len(frame), _p(out, _u8p), out.size)
    return out[:n].tobytes()


class FreqShiftBatch:
    """rows x cFreqShift (FreqShift.h:12-27): one float32 NCO per row, never wrapped (x86 reference behaviour)."""

    def __init__(self, nco_freq, in_rate: float, max_len: int = 65536, device: int = -1):
        f = np.ascontiguousarray(np.atleast_1d(nco_freq), dtype=np.float32)
        self.rows = f.size
        self._h = C.c_void_p()
        _check(lib().rfm_freqshift_create(self.rows, _p(f, _f32p), in_rate, max_len, device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_freqshift_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        _check(lib().rfm_freqshift_reset(self._h))

    def process_cf32(self, iq: np.ndarray) -> np.ndarray:
        iq = np.array(iq, dtype=np.float32, order="C").reshape(self.rows, -1, 2)
        _check(lib().rfm_freqshift_process_cf32(self._h, _p(iq, _f32p), iq.shape[1]))
        return iq

    def process_u8(self, iq_u8: np.ndarray, shared_capture: bool) -> np.ndarray:
        iq_u8 = np.ascontiguousarray(iq_u8, dtype=np.uint8)
        n = iq_u8.reshape(-1, 2).shape[0] // (1 if shared_capture else self.rows)
        out = np.empty((self.rows, n, 2), dtype=np.float32)
        _check(lib().rfm_freqshift_process_u8(self._h, _p(iq_u8, _u8p), int(shared_capture), n, _p(out, _f32p)))
        return out

    def process_iq(self, iq: np.ndarray, shared_capture: bool) -> np.ndarray:
        """iq of uint8 / int8 / int16 / float32 (complex64): one capture [n, 2] shared by every row, or [rows, n, 2] ->
        out [rows, n, 2] float32."""
        fmt, iq = _iq_host(iq)
        n = iq.shape[0] // (1 if shared_capture else self.rows)
        out = np.empty((self.rows, n, 2), dtype=np.float32)
        _check(lib().rfm_freqshift_process_iq(self._h, fmt, int(shared_capture), iq.ctypes.data_as(C.c_void_p), n,
                                              _p(out, _f32p)))
        return out

    def process_iq_device(self, fmt, shared_capture: bool, d_in_ptr: int, in_stride: int, d_out_ptr: int, out_stride: int,
                          n: int, cuda_stream: int = 0):
        _check(lib().rfm_freqshift_process_iq_device(self._h, iq_format(fmt), int(shared_capture), C.c_void_p(d_in_ptr),
                                                     in_stride, C.c_void_p(d_out_ptr), out_stride, n,
                                                     C.c_void_p(cuda_stream)))

    def set_iq_correction(self, c: IqCorrection | None):
        """IQ correction of every later process call (None = off)."""
        _check(lib().rfm_freqshift_set_iq_correction(self._h, _corr_arg(c)))

    def process_device(self, mode: int, d_in_ptr: int, in_stride: int, d_out_ptr: int, out_stride: int, n: int,
                       cuda_stream: int = 0):
        _check(lib().rfm_freqshift_process_device(self._h, mode, C.c_void_p(d_in_ptr), in_stride, C.c_void_p(d_out_ptr),
                                                  out_stride, n, C.c_void_p(cuda_stream)))


class DownConvertBatch:
    """rows x CRDSDownConvert (DownConvert.h:68-169): NCO_OSC mixer + decimate-by-2 chain, one row per station / stream."""

    def __init__(self, nco_freq, in_rate: float, max_bw: float, wfm: bool = False, max_len: int = 65536, device: int = -1):
        f = np.ascontiguousarray(np.atleast_1d(nco_freq), dtype=np.float32)
        self.rows = f.size
        self._h = C.c_void_p()
        _check(lib().rfm_downconvert_create(self.rows, _p(f, _f32p), in_rate, max_bw, int(wfm), max_len, device,
                                            C.byref(self._h)))
        taps = np.zeros(16, dtype=np.uint32)
        self.n_stages = int(lib().rfm_downconvert_stages(self._h, _p(taps, _u32p), 16))
        self.stage_taps = taps[:self.n_stages].tolist()
        self.output_rate = float(lib().rfm_downconvert_output_rate(self._h))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_downconvert_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        _check(lib().rfm_downconvert_reset(self._h))

    def set_frequency(self, nco_freq):
        f = np.ascontiguousarray(np.atleast_1d(nco_freq), dtype=np.float32)
        assert f.size == self.rows
        _check(lib().rfm_downconvert_set_frequency(self._h, _p(f, _f32p)))

    def set_premix(self, d_table_ptr: int, row_stride: int, period: int):
        """Device table [rows][row_stride] float2 of a cFreqShift that is Reset() every `period` samples (0 = off)."""
        _check(lib().rfm_downconvert_set_premix(self._h, C.c_void_p(d_table_ptr) if d_table_ptr else None, row_stride,
                                                period))

    def set_iq_correction(self, c: IqCorrection | None):
        """IQ correction of every later process call, before the pre-mix table and the NCO (None = off)."""
        _check(lib().rfm_downconvert_set_iq_correction(self._h, _corr_arg(c)))

    def set_nco(self, nco_freq):
        """Phase-accumulator NCO pre-mixer (rfm_downconvert_set_nco): one frequency per row in Hz, |f| <= in_rate / 2,
        every phase restarted at 0; None switches it off.  Pass -f to bring a station at +f to 0 Hz."""
        if nco_freq is None:
            _check(lib().rfm_downconvert_set_nco(self._h, None))
            return
        f = np.ascontiguousarray(np.atleast_1d(nco_freq), dtype=np.float64)
        if f.size != self.rows:
            raise ValueError(f"{f.size} frequencies for {self.rows} rows")
        _check(lib().rfm_downconvert_set_nco(self._h, _p(f, _f64p)))

    def process_cf32(self, iq: np.ndarray) -> np.ndarray:
        iq = np.ascontiguousarray(iq, dtype=np.float32).reshape(self.rows, -1, 2)
        n = iq.shape[1]
        out = np.empty((self.rows, max(n >> self.n_stages, 1), 2), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_downconvert_process_cf32(self._h, _p(iq, _f32p), n, _p(out, _f32p), C.byref(k)))
        return out[:, :k.value].copy()

    def process_u8(self, iq_u8: np.ndarray, shared_capture: bool) -> np.ndarray:
        iq_u8 = np.ascontiguousarray(iq_u8, dtype=np.uint8)
        n = iq_u8.reshape(-1, 2).shape[0] // (1 if shared_capture else self.rows)
        out = np.empty((self.rows, max(n >> self.n_stages, 1), 2), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_downconvert_process_u8(self._h, _p(iq_u8, _u8p), int(shared_capture), n, _p(out, _f32p),
                                                C.byref(k)))
        return out[:, :k.value].copy()

    def process_iq(self, iq: np.ndarray, shared_capture: bool) -> np.ndarray:
        """iq of uint8 / int8 / int16 / float32 (complex64): one capture [n, 2] shared by every row, or [rows, n, 2] ->
        out [rows, n >> stages, 2] float32."""
        fmt, iq = _iq_host(iq)
        n = iq.shape[0] // (1 if shared_capture else self.rows)
        out = np.empty((self.rows, max(n >> self.n_stages, 1), 2), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_downconvert_process_iq(self._h, fmt, int(shared_capture), iq.ctypes.data_as(C.c_void_p), n,
                                                _p(out, _f32p), C.byref(k)))
        return out[:, :k.value].copy()

    def process_iq_device(self, fmt, shared_capture: bool, d_in_ptr: int, in_stride: int, d_out_ptr: int,
                          out_stride: int, n: int, cuda_stream: int = 0) -> int:
        k = C.c_uint32(0)
        _check(lib().rfm_downconvert_process_iq_device(self._h, iq_format(fmt), int(shared_capture), C.c_void_p(d_in_ptr),
                                                       in_stride, C.c_void_p(d_out_ptr), out_stride, n, C.byref(k),
                                                       C.c_void_p(cuda_stream)))
        return int(k.value)

    def process_device(self, mode: int, d_in_ptr: int, in_stride: int, d_out_ptr: int, out_stride: int, n: int,
                       cuda_stream: int = 0) -> int:
        k = C.c_uint32(0)
        _check(lib().rfm_downconvert_process_device(self._h, mode, C.c_void_p(d_in_ptr), in_stride, C.c_void_p(d_out_ptr),
                                                    out_stride, n, C.byref(k), C.c_void_p(cuda_stream)))
        return int(k.value)


class _RowFilter:
    """Common part of IirFilterBatch / FirFilterBatch: in-place Process / ProcessTwo on host arrays [rows, n(, 2)]."""
    _kind = ""

    def __init__(self, rows: int, max_len: int = 65536, device: int = -1):
        self.rows = rows
        self._h = C.c_void_p()
        _check(getattr(lib(), f"rfm_{self._kind}_create")(rows, max_len, device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            getattr(lib(), f"rfm_{self._kind}_destroy")(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def process_real(self, x: np.ndarray) -> np.ndarray:
        x = np.array(x, dtype=np.float32, order="C").reshape(self.rows, -1)
        _check(getattr(lib(), f"rfm_{self._kind}_process_real")(self._h, _p(x, _f32p), x.shape[1]))
        return x

    def process_complex(self, x: np.ndarray) -> np.ndarray:
        x = np.array(x, dtype=np.float32, order="C").reshape(self.rows, -1, 2)
        _check(getattr(lib(), f"rfm_{self._kind}_process_complex")(self._h, _p(x, _f32p), x.shape[1]))
        return x

    def process_two(self, a: np.ndarray, b: np.ndarray):
        a = np.array(a, dtype=np.float32, order="C").reshape(self.rows, -1)
        b = np.array(b, dtype=np.float32, order="C").reshape(self.rows, -1)
        _check(getattr(lib(), f"rfm_{self._kind}_process_two")(self._h, _p(a, _f32p), _p(b, _f32p), a.shape[1]))
        return a, b


class IirFilterBatch(_RowFilter):
    """rows x cIirFilter (IirFilter.h:12-36).  type: 0 LP, 1 HP, 2 BP, 3 BR."""
    _kind = "iir"

    def init(self, ftype: int, f0: float, q: float, fs: float) -> bool:
        rc = lib().rfm_iir_init(self._h, ftype, f0, q, fs)
        if rc == -1:
            return False            # cIirFilter::Init returns false for an unknown type
        _check(rc)
        return True

    def coefficients(self) -> np.ndarray:
        out = np.zeros(5, dtype=np.float32)
        _check(lib().rfm_iir_coefficients(self._h, _p(out, _f32p)))
        return out


def fir_design(kind: str, num_taps: int, scale: float, astop: float, fpass: float, fstop: float, fs: float) -> np.ndarray:
    """Taps of cFirFilter::InitLPFilter (kind "lp", FirFilter.cpp:78-148) / InitHPFilter ("hp", :195-264); host only."""
    out = np.zeros(128, dtype=np.float32)
    k = C.c_uint32(0)
    _check(lib().rfm_fir_design({"lp": 0, "hp": 1}[kind], num_taps, scale, astop, fpass, fstop, fs, _p(out, _f32p),
                                out.size, C.byref(k)))
    return out[:k.value].copy()


class FirFilterBatch(_RowFilter):
    """rows x cFirFilter (FirFilter.h:17-60)."""
    _kind = "fir"

    def init_lp(self, num_taps: int, scale: float, astop: float, fpass: float, fstop: float, fs: float) -> int:
        k = C.c_uint32(0)
        _check(lib().rfm_fir_init_lp(self._h, num_taps, scale, astop, fpass, fstop, fs, C.byref(k)))
        return int(k.value)

    def init_hp(self, num_taps: int, scale: float, astop: float, fpass: float, fstop: float, fs: float) -> int:
        """cFirFilter::InitHPFilter (FirFilter.cpp:195-264)."""
        k = C.c_uint32(0)
        _check(lib().rfm_fir_init_hp(self._h, num_taps, scale, astop, fpass, fstop, fs, C.byref(k)))
        return int(k.value)

    def init_const(self, coef, fs: float):
        c = np.ascontiguousarray(coef, dtype=np.float32)
        _check(lib().rfm_fir_init_const(self._h, c.size, _p(c, _f32p), fs))

    def taps(self) -> np.ndarray:
        out = np.zeros(128, dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_fir_taps(self._h, _p(out, _f32p), out.size, C.byref(k)))
        return out[:k.value].copy()


class DownsampleFilterBatch:
    """rows x cDownsampleFilter (DownConvert.h:21-60): complex + integer factor, real + fractional or integer factor."""

    def __init__(self, rows: int, filter_order: int, cutoff: float, downsample: float = 1.0, integer_factor: bool = True,
                 max_len: int = 65536, device: int = -1):
        self.rows = rows
        self._h = C.c_void_p()
        _check(lib().rfm_downsample_create(rows, filter_order, cutoff, downsample, int(integer_factor), max_len, device,
                                           C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_downsample_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        _check(lib().rfm_downsample_reset(self._h))

    def coefficients(self) -> np.ndarray:
        out = np.zeros(1024, dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_downsample_coefficients(self._h, _p(out, _f32p), out.size, C.byref(k)))
        return out[:k.value].copy()

    def process_complex(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.rows, -1, 2)
        n = x.shape[1]
        out = np.zeros((self.rows * int(lib().rfm_downsample_max_outputs(self._h, n)), 2), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_downsample_process_complex(self._h, _p(x, _f32p), _p(out, _f32p), n, C.byref(k)))
        return out[:self.rows * k.value].reshape(self.rows, k.value, 2).copy()

    def process_real(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float32).reshape(self.rows, -1)
        n = x.shape[1]
        out = np.zeros(self.rows * int(lib().rfm_downsample_max_outputs(self._h, n)), dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_downsample_process_real(self._h, _p(x, _f32p), _p(out, _f32p), n, C.byref(k)))
        return out[:self.rows * k.value].reshape(self.rows, k.value).copy()


class RdsProcessorBatch:
    """rows x cRDSRxSignalProcessor (RDSProcess.h:56-110): FM baseband in, RDS bits / groups out."""

    def __init__(self, rows: int, sample_rate: float, max_len: int = 65536, device: int = -1):
        self.rows = rows
        self._h = C.c_void_p()
        _check(lib().rfm_rdsproc_create(rows, sample_rate, max_len, device, C.byref(self._h)))
        self.process_rate = float(lib().rfm_rdsproc_process_rate(self._h))

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_rdsproc_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def reset(self):
        _check(lib().rfm_rdsproc_reset(self._h))

    def process(self, baseband: np.ndarray):
        x = np.ascontiguousarray(baseband, dtype=np.float32).reshape(self.rows, -1)
        _check(lib().rfm_rdsproc_process(self._h, _p(x, _f32p), x.shape[1]))

    def take_bits(self, row: int = 0, max_bits: int = 1 << 20) -> np.ndarray:
        out = np.zeros(max_bits, dtype=np.uint8)
        k = C.c_uint32(0)
        _check(lib().rfm_rdsproc_take_bits(self._h, row, _p(out, _u8p), max_bits, C.byref(k)))
        return out[:k.value].copy()

    def take_groups(self, row: int = 0, max_groups: int = 4096) -> np.ndarray:
        out = np.zeros((max_groups, 4), dtype=np.uint16)
        k = C.c_uint32(0)
        _check(lib().rfm_rdsproc_take_groups(self._h, row, _p(out, _u16p), max_groups, C.byref(k)))
        return out[:k.value].copy()


SCAN_BINS = 4096


def scan_config(fs: float, raster_first: float, raster_step: float, raster_count: int, min_snr_db: float = 10.0,
                device: int = -1) -> ScanConfig:
    cfg = ScanConfig()
    lib().rfm_scan_config_default(C.byref(cfg))
    cfg.sample_rate, cfg.raster_first, cfg.raster_step = fs, raster_first, raster_step
    cfg.raster_count, cfg.min_snr_db, cfg.device = raster_count, min_snr_db, device
    return cfg


SCAN_MIXERS = {"osc": 0, "nco": 1}   # rfm_scan_set_mixer: RFM_SCAN_MIXER_OSC, RFM_SCAN_MIXER_NCO


def scan_mixer(mixer: str) -> int:
    """The confirmation's mixer: "osc" (CRDSDownConvert's NCO_OSC at -f_j) or "nco" (rows at 0 Hz behind the phasor
    NCO); ValueError otherwise."""
    if not isinstance(mixer, str) or mixer not in SCAN_MIXERS:
        raise ValueError(f"unknown scan mixer {mixer!r}: use \"osc\" or \"nco\"")
    return SCAN_MIXERS[mixer]


class BandScan:
    """Band scan of one wideband capture (rfm_scan_*; u8, s8, s16 or cf32): averaged spectrum, channel powers on a raster (Hz from the
    capture centre), candidates, and every candidate confirmed with the reference's receiver -- the add-on's tuner
    auto-scan (ChannelSettings.cpp:96-147) for all channels at once.  mixer = "nco" confirms with the phase-accumulator
    NCO in front of rows at 0 Hz instead of CRDSDownConvert's NCO_OSC ("osc", the default)."""

    def __init__(self, fs: float, raster_first: float, raster_step: float, raster_count: int, min_snr_db: float = 10.0,
                 device: int = -1, iq_correction=None, mixer: str = "osc"):
        mixer_id = scan_mixer(mixer)
        cfg = scan_config(fs, raster_first, raster_step, raster_count, min_snr_db, device)
        self.raster_count = raster_count
        self._h = C.c_void_p()
        _check(lib().rfm_scan_create(C.byref(cfg), C.byref(self._h)))
        self.set_iq_correction(iq_correction)
        _check(lib().rfm_scan_set_mixer(self._h, mixer_id))

    def set_iq_correction(self, c):
        """IQ correction of later runs: None (off), "estimate" (from each run's capture) or a fixed IqCorrection."""
        if c is None:
            _check(lib().rfm_scan_set_iq_correction(self._h, 0, None))
        elif isinstance(c, str):
            if c != "estimate":
                raise ValueError(f"unknown IQ correction mode {c!r}: use None, \"estimate\" or an IqCorrection")
            _check(lib().rfm_scan_set_iq_correction(self._h, 1, None))
        else:
            _check(lib().rfm_scan_set_iq_correction(self._h, 2, _corr_arg(c)))

    def iq_correction(self) -> IqCorrection:
        """The correction the last run applied (identity with imbalance_valid False when off)."""
        out = RfmIqCorrection()
        _check(lib().rfm_scan_iq_correction(self._h, C.byref(out)))
        return IqCorrection._from_c(out)

    def close(self):
        if getattr(self, "_h", None):
            lib().rfm_scan_destroy(self._h)
            self._h = None

    __del__ = _quiet_del(close)

    def run_u8(self, capture_u8: np.ndarray):
        """Host capture [n, 2] uint8."""
        cap = np.ascontiguousarray(capture_u8, dtype=np.uint8).reshape(-1, 2)
        _check(lib().rfm_scan_run_u8(self._h, cap.ctypes.data_as(C.c_void_p), cap.shape[0], 0))

    def run(self, capture):
        """capture: a host array [n, 2] of uint8 / int8 / int16 / float32 ([n] complex64), or a CUDA tensor of those
        dtypes, complete before the call (e.g. after torch.cuda.synchronize()).  The format comes from the dtype."""
        if hasattr(capture, "data_ptr") and getattr(capture, "is_cuda", False):
            fmt = iq_format(capture.dtype)
            if not capture.is_contiguous():
                raise ValueError("device capture must be contiguous")
            n = capture.numel() // (1 if fmt == IQ_CF32 and capture.is_complex() else 2)
            _check(lib().rfm_scan_run(self._h, fmt, C.c_void_p(capture.data_ptr()), n, 1))
            return
        fmt, cap = _iq_host(capture)
        _check(lib().rfm_scan_run(self._h, fmt, cap.ctypes.data_as(C.c_void_p), cap.shape[0], 0))

    def run_device(self, d_capture_ptr: int, n: int):
        """Device capture [n, 2] uint8 at d_capture_ptr, complete before the call (e.g. after torch.cuda.synchronize())."""
        _check(lib().rfm_scan_run_u8(self._h, C.c_void_p(d_capture_ptr), n, 1))

    def spectrum(self) -> np.ndarray:
        out = np.zeros(SCAN_BINS, dtype=np.float32)
        k = C.c_uint32(0)
        _check(lib().rfm_scan_spectrum(self._h, _p(out, _f32p), out.size, C.byref(k)))
        return out[:k.value]

    def channel_power(self) -> np.ndarray:
        out = np.zeros(self.raster_count, dtype=np.float64)
        _check(lib().rfm_scan_channel_power(self._h, _p(out, _f64p), out.size))
        return out

    def stations(self) -> list[dict]:
        n = C.c_uint32(0)
        buf = (ScanStation * self.raster_count)()          # at most one station per channel
        _check(lib().rfm_scan_stations(self._h, buf, len(buf), C.byref(n)))
        return [scan_station_dict(buf[i]) for i in range(n.value)]

    def timing(self) -> tuple[float, float]:
        """(spectrum, confirmation) device milliseconds of the last run."""
        a, b = C.c_double(0), C.c_double(0)
        _check(lib().rfm_scan_timing(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value


def scan_station_dict(st: ScanStation) -> dict:
    return {"freq": st.freq, "power_dbfs": np.float32(st.power_dbfs), "snr_db": np.float32(st.snr_db),
            "stereo": bool(st.stereo_detected), "pilot_level": np.float32(st.pilot_level),
            "if_level": np.float32(st.interface_level), "bb_level": np.float32(st.baseband_level),
            "rds_groups": int(st.rds_groups), "pi": int(st.pi), "ps": st.ps.decode("latin-1")}


def math_probe(op: int, a: np.ndarray, b: np.ndarray | None = None) -> np.ndarray:
    """Evaluate a scalar building block of the kernels on the device; returns [n, 2] float32 (see radiofm_b200.h)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    out = np.zeros((a.size, 2), dtype=np.float32)
    pb = None
    if b is not None:
        b = np.ascontiguousarray(b, dtype=np.float32)
        assert b.size == a.size
        pb = _p(b, _f32p)
    _check(lib().rfm_math_probe(op, _p(a, _f32p), pb, _p(out, _f32p), a.size))
    return out


def div_selftest(pairs: int, seed: int = 1) -> tuple[int, int]:
    m, t = C.c_uint64(0), C.c_uint64(0)
    _check(lib().rfm_div_selftest(seed, pairs, C.byref(m), C.byref(t)))
    return int(m.value), int(t.value)


def rds_check_block(word26: int, offset_syndrome: int, use_fec: bool):
    c = C.c_uint32(0)
    syn = lib().rfm_rds_check_block(word26, offset_syndrome, int(use_fec), C.byref(c))
    return int(syn), int(c.value)
