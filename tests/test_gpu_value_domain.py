"""Every chain against the oracle at the edges of the sample-value domain (the classes of test_value_domain.py: zero
runs, rail codes, extreme and subnormal cf32 magnitudes, NaN and Inf), bit for bit.

The contract: for finite input every output is the oracle's, bit for bit (the oracle fed to_cf32 of the same samples);
where the oracle's own arithmetic makes a NaN (a non-finite sample, or an overflow inside the chain) the outputs are
NaN-equivalent (NaN at the same places, every other value bit-equal: x86 and the GPU make different NaN bit patterns),
a stream's NaN stays in that stream, and reset() clears what cFmDecoder::Reset clears, no more.  The band scan
refuses a spectrum with a non-finite bin.  test_value_domain.py::test_value_classes_reach_every_replay_family shows on the CPU that these
inputs reach the lane kernels' replay paths.

Loops and indices whose bounds could come from sample values, in the kernels these cases reach: the front ends, the
down-converter and the scan index by sample position only.  The exact wraps (rfm_wrap_demod's `while (phase < 0)`,
rfm_fmod_2pi_small's `while (r >= 2 pi)`) would not end for an infinite phase; the demodulator's phase is the sum of
a clamped increment and alpha * err with |err| <= pi, so it is finite or NaN, and NaN fails both conditions.  The
pilot's frequency is clamped by selects that turn a NaN into a limit.  The repair passes are bounded by the chunk count.
"""
from __future__ import annotations

import importlib

import numpy as np
import pytest

from conftest import RATES, bits_equal, station
from oracle import iqcorr, nco as onco, scan
from test_iq_formats import to_cf32, welch_psd_iq
from test_kernel_instantiations import _rds_skipped_blocks, _rds_stage_lengths
from test_value_domain import (M_EXPONENTS, N_BLOCKS, assert_subnormals_kept, decoder_classes, every_code, nan_equal,
                               non_finite, ramp_across, requantise, scaled, with_rails, with_zero_runs)

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


@pytest.fixture(autouse=True)
def _subnormals_kept():
    assert_subnormals_kept()


def _same_status(a: dict, b: dict) -> bool:
    return all(nan_equal(np.atleast_1d(np.float32(a[k])), np.atleast_1d(np.float32(b[k]))) for k in b)


# ---------------------------------------------------------------------------------------------------------------------
# decoder
# ---------------------------------------------------------------------------------------------------------------------
DECODERS = {   # label -> (synthetic station / block length, fs, downsample)
    "2.4M/11": ("2.4M", 2.4e6, 11),      # s8 rows on the TMA front end
    "1.0M/4": ("1.0M", 1.0e6, 4),        # tiled front end
    "1.0M/3": ("1.0M", 1.0e6, 3),        # generic k_front
    "390k/1": ("390k", 390625.0, 1),
}
ENTRIES = ("host", "submit", "device")


class _Run:
    """One FmDecoderBatch fed through one entry point, block by block."""

    def __init__(self, rfm, label, entry, S, blk):
        _, fs, ds = DECODERS[label]
        self.torch, self.entry, self.S = _torch(), entry, S
        self.d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=S, max_block_len=blk, device=0)
        self.stride = (self.d.max_audio_floats(blk) + 1) & ~1

    def block(self, x: np.ndarray, fmt: str) -> np.ndarray:
        if self.entry == "host":
            return self.d.process_iq(x)
        if self.entry == "submit":
            a = self.d.process_iq(x, submit=True)
            self.d.synchronize()
            return a.copy()
        torch = self.torch
        t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        a = torch.empty((self.S, self.stride), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        k = self.d.process_iq_device(fmt, t.data_ptr(), x.shape[1], x.shape[1], a.data_ptr(), self.stride)
        self.d.synchronize()
        return a[:, :k].cpu().numpy()

    def outputs(self, s):
        return self.d.take_bits(s), self.d.take_groups(s), self.d.status(s)


def _compare_rds(rfm, label: str, blk: int) -> bool:
    """False where a block skips the RDS branch (odd counts into a fixed stage, DESIGN.md section 7): the oracle's
    bits are not comparable after it."""
    return not _rds_skipped_blocks(_rds_stage_lengths(rfm, label), DECODERS[label][2], [blk] * N_BLOCKS)


def _batch(label: str, fmt: str):
    rate, _, ds = DECODERS[label]
    cls = decoder_classes(rate, fmt, ds)
    return list(cls), np.stack(list(cls.values()))


@pytest.mark.parametrize("fmt", ["s8", "s16", "cf32"])
@pytest.mark.parametrize("label", list(DECODERS))
def test_decoder_value_classes(rfm, port, label, fmt):
    """One class per stream (stream 0 a clean station) through the host, submit and device entry points: audio, the
    baseband tap, status, RDS bits and groups against port.OracleFmDecoder block by block.  Then isolation: the same
    batch with every odd stream replaced by a clean station leaves every even stream's outputs bit-identical."""
    rate, fs, ds = DECODERS[label]
    blk = RATES[rate][2]
    names, raw = _batch(label, fmt)
    S = len(names)
    oracles = [port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds) for _ in range(S)]
    runs = {e: _Run(rfm, label, e, S, blk) for e in ENTRIES}
    clean = raw.copy()
    clean[1::2] = raw[0]
    iso = _Run(rfm, label, "host", S, blk)
    iso_audio, host_audio = [], []
    for b in range(N_BLOCKS):
        x = np.ascontiguousarray(raw[:, b * blk:(b + 1) * blk])
        want = [o.process_cf32(to_cf32(x[s])) for s, o in enumerate(oracles)]
        want_bb = [o.tap("baseband") for o in oracles]
        for e, r in runs.items():
            got = r.block(x, fmt)
            for s in range(S):
                assert nan_equal(got[s], want[s]), (label, fmt, e, b, names[s], "audio")
                assert nan_equal(r.d.tap("baseband", s), want_bb[s]), (label, fmt, e, b, names[s], "baseband")
            if e == "host":
                host_audio.append(got)
        iso_audio.append(iso.block(np.ascontiguousarray(clean[:, b * blk:(b + 1) * blk]), fmt))
    rds = _compare_rds(rfm, label, blk)
    for s, o in enumerate(oracles):
        bits, groups, st = o.take_bits(), o.take_groups(), o.status()
        assert bits.size > 0 or s > 0, (label, fmt)
        for e, r in runs.items():
            gb, gg, gs = r.outputs(s)
            same_rds = np.array_equal(gb, bits) and np.array_equal(gg, groups)
            assert same_rds or not rds, (label, fmt, e, names[s], "RDS")
            assert _same_status(gs, st), (label, fmt, e, names[s], gs, st)
        o.close()
    for s in range(0, S, 2):
        for b in range(N_BLOCKS):
            assert bits_equal(iso_audio[b][s], host_audio[b][s]), (label, fmt, "isolation", b, names[s])
    for r in list(runs.values()) + [iso]:
        r.d.close()


NF_KINDS = ("nan", "inf", "nan32")


@pytest.mark.parametrize("label", ["1.0M/4", "2.4M/11"])
def test_decoder_non_finite_stream(rfm, port, label):
    """Streams 1..3 carry a NaN sample, an +Inf sample and a 32-sample NaN burst in block 2.  Every call returns
    RFM_OK; blocks before the first bad sample are bit-exact, the rest NaN-equivalent to the oracle; stream 0 (clean)
    is bit-exact throughout.  reset() is cFmDecoder::Reset (FmDecode.cpp:326-338): the meters, the demodulator PLL
    and RDS start over, the filters' delay lines and the de-emphasis state do not, so a NaN held there stays -- in the
    reference too.  After it, against the oracles reset the same way, stream 0 stays bit-exact and the others
    NaN-equivalent."""
    rate, fs, ds = DECODERS[label]
    blk = RATES[rate][2]
    base = requantise(station(rate, N_BLOCKS, stream_id=42)[0][:N_BLOCKS * blk], "cf32")
    rows, first = [requantise(station(rate, N_BLOCKS, stream_id=40)[0][:N_BLOCKS * blk], "cf32")], [None]
    for kind in NF_KINDS:
        y, p = non_finite(base, blk, kind)
        rows.append(y)
        first.append(p)
    raw = np.stack(rows)
    S = raw.shape[0]
    oracles = [port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds) for _ in range(S)]
    runs = {e: _Run(rfm, label, e, S, blk) for e in ENTRIES}
    saw_nan = False
    for b in range(N_BLOCKS):
        x = np.ascontiguousarray(raw[:, b * blk:(b + 1) * blk])
        want = [o.process_cf32(x[s]) for s, o in enumerate(oracles)]
        want_bb = [o.tap("baseband") for o in oracles]
        for e, r in runs.items():
            got = r.block(x, "cf32")                     # raises RadioFmError on anything but RFM_OK
            for s in range(S):
                clean = first[s] is None or (b + 1) * blk <= first[s]
                same = bits_equal if clean else nan_equal
                assert same(got[s], want[s]), (label, e, b, s, "audio")
                assert same(r.d.tap("baseband", s), want_bb[s]), (label, e, b, s, "baseband")
                saw_nan |= bool(np.isnan(got[s]).any())
    assert saw_nan
    assert _compare_rds(rfm, label, blk)
    for s, o in enumerate(oracles):
        bits, groups, st = o.take_bits(), o.take_groups(), o.status()
        for e, r in runs.items():
            gb, gg, gs = r.outputs(s)
            assert np.array_equal(gb, bits) and np.array_equal(gg, groups), (label, e, s, "RDS")
            assert _same_status(gs, st), (label, e, s, gs, st)
    # reset, then clean stations in every stream
    fresh = np.stack([requantise(station(rate, 2, stream_id=50 + s)[0][:2 * blk], "cf32") for s in range(S)])
    for o in oracles:
        o.reset()
    for r in runs.values():
        r.d.reset()
        for s in range(S):
            r.outputs(s)                                 # drop what the bad run left queued
    for b in range(2):
        x = np.ascontiguousarray(fresh[:, b * blk:(b + 1) * blk])
        want = [o.process_cf32(x[s]) for s, o in enumerate(oracles)]
        for e, r in runs.items():
            got = r.block(x, "cf32")
            for s in range(S):
                assert (bits_equal if s == 0 else nan_equal)(got[s], want[s]), (label, e, "after reset", b, s)
    for s, o in enumerate(oracles):
        bits, groups, st = o.take_bits(), o.take_groups(), o.status()
        for e, r in runs.items():
            gb, gg, gs = r.outputs(s)
            assert np.array_equal(gb, bits) and np.array_equal(gg, groups), (label, e, "after reset", s, "RDS")
            assert _same_status(gs, st), (label, e, "after reset", s, gs, st)
        o.close()
    for r in runs.values():
        r.d.close()


# ---------------------------------------------------------------------------------------------------------------------
# wideband front end
# ---------------------------------------------------------------------------------------------------------------------
FS, BLK, BPC = 50.0e6, 32000, 64
N_WIDE = 6 * BLK
CALLS = (24 * 5120, N_WIDE - 24 * 5120)              # the uniform HB51 chain's tiles; both multiples of 2^7
FREQS = [-1.0e6, 200000.0, 7.0e6]


@pytest.fixture(scope="module")
def wide_u8(synth):
    return synth.make_wideband_u8(FS, N_WIDE, FREQS)


def _wide_classes(u8: np.ndarray, fmt: str) -> dict[str, np.ndarray]:
    x = requantise(u8, fmt, seed=9)
    out = {"Z": with_zero_runs(x, BLK, 1)}
    if fmt == "cf32":
        for k in M_EXPONENTS:
            out[f"M 2^{k}"] = scaled(x, k)
        out["M ramp 2^-95"] = ramp_across(x, BLK)
    else:
        out["R"] = with_rails(x, BLK)
        out["R +6 dB clipped"] = requantise(u8, fmt, seed=9, gain=2.0)
        out["R every code"] = every_code(fmt, N_WIDE, seed=3)
    return out


class _OracleDc:
    def __init__(self, port, freq):
        import ctypes as C
        self.C, self.L = C, port.lib()
        self.h = self.L.rfo_rdsdc_create()
        self.L.rfo_rdsdc_set_frequency(self.h, np.float32(freq))
        self.L.rfo_rdsdc_set_wfm_data_rate(self.h, np.float32(FS), np.float32(100000.0))

    def process(self, x):
        P = lambda a: a.ctypes.data_as(self.C.POINTER(self.C.c_float))   # noqa: E731
        z = np.array(x, dtype=np.float32, order="C").reshape(-1, 2)
        y = np.zeros_like(z)
        k = self.L.rfo_rdsdc_process(self.h, z.shape[0], P(z), P(y))
        return y[:k].copy()

    def close(self):
        self.L.rfo_rdsdc_destroy(self.h)


def _freqshift_blocks(port, f, x, period):
    """cFreqShift(f) reset every `period` samples (the pre-mix table's and the receiver's use), on float samples."""
    import ctypes as C
    L = port.lib()
    h = L.rfo_freqshift_create(np.float32(f), np.float32(FS))
    y = np.array(x, dtype=np.float32, order="C").reshape(-1, 2)
    for p in range(0, y.shape[0], period):
        z = np.ascontiguousarray(y[p:p + period])
        L.rfo_freqshift_reset(h)
        L.rfo_freqshift_process(h, z.ctypes.data_as(C.POINTER(C.c_float)), z.shape[0])
        y[p:p + period] = z
    L.rfo_freqshift_destroy(h)
    return y


@pytest.mark.parametrize("corr", [False, True])
@pytest.mark.parametrize("fmt", ["s8", "s16", "cf32"])
def test_wideband_mixers_value_classes(rfm, port, wide_u8, fmt, corr):
    """DownConvertBatch with the osc, a pre-mix table and the NCO, and FreqShiftBatch, on shared captures of the value
    classes, host and device entry points, against the oracle's CRDSDownConvert and cFreqShift on cf32 rows (IQ
    correction: the capture's own estimate, applied by oracle/iqcorr.apply).  cFreqShift restarts every call (every
    front-end block for the table), so its float phase stays below 2 pi f 32000 / Fs < 1e5."""
    torch = _torch()
    dev = torch.device("cuda", 0)
    ones = np.zeros((3, BLK, 2), dtype=np.float32)
    ones[:, :, 0] = 1.0
    fsb = rfm.FreqShiftBatch([-f for f in FREQS], FS, max_len=BLK, device=0)
    table = torch.from_numpy(fsb.process_cf32(ones)).to(dev)
    fsb.close()
    for name, raw in _wide_classes(wide_u8, fmt).items():
        x = to_cf32(raw)
        c = rfm.estimate_iq_correction(raw) if corr else None
        if corr:
            assert np.isfinite([c.dc_i, c.dc_q, c.a, c.b]).all(), (name, c)
            x = iqcorr.apply(x, c.dc_i, c.dc_q, c.a, c.b)
        for mixer in ("osc", "premix", "nco"):
            d = rfm.DownConvertBatch([-f for f in FREQS] if mixer == "osc" else [0.0] * 3, FS, 100000.0, wfm=True,
                                     max_len=max(CALLS), device=0)
            if corr:
                d.set_iq_correction(c)
            if mixer == "premix":
                d.set_premix(table.data_ptr(), BLK, BLK)
            if mixer == "nco":
                d.set_nco([-f for f in FREQS])
            ncos = [onco.Nco(-f, np.float32(FS)) for f in FREQS]
            oracles = [_OracleDc(port, -f if mixer == "osc" else 0.0) for f in FREQS]
            pos = 0
            for i, n in enumerate(CALLS):
                seg = slice(pos, pos + n)
                m = n >> d.n_stages
                if i == 0:
                    got = d.process_iq(raw[seg], shared_capture=True)
                else:
                    t = torch.from_numpy(np.ascontiguousarray(raw[seg])).to(dev)
                    out = torch.empty((3, m, 2), dtype=torch.float32, device=dev)
                    assert d.process_iq_device(fmt, True, t.data_ptr(), 0, out.data_ptr(), m, n) == m
                    torch.cuda.synchronize()
                    got = out.cpu().numpy()
                for r, f in enumerate(FREQS):
                    xr = x[seg]
                    if mixer == "premix":
                        xr = _freqshift_blocks(port, -f, x, BLK)[seg]
                    elif mixer == "nco":
                        xr = ncos[r].mix(xr)
                    assert nan_equal(got[r], oracles[r].process(xr)), (fmt, corr, name, mixer, i, r)
                pos += n
            for o in oracles:
                o.close()
            d.close()
        # FreqShiftBatch, one call per front-end block, reset before each (as the receiver uses cFreqShift)
        fs = rfm.FreqShiftBatch([-f for f in FREQS], FS, max_len=BLK, device=0)
        if corr:
            fs.set_iq_correction(c)
        for b in (0, 3, 4):
            fs.reset()
            got = fs.process_iq(np.ascontiguousarray(raw[b * BLK:(b + 1) * BLK]), shared_capture=True)
            for r, f in enumerate(FREQS):
                want = _freqshift_blocks(port, -f, x[b * BLK:(b + 1) * BLK], BLK)
                assert nan_equal(got[r], want), (fmt, corr, name, "freqshift", b, r)
        fs.close()


@pytest.mark.parametrize("fmt,cls,mixer", [("s16", "R +6 dB clipped", "osc"), ("cf32", "M 2^-100", "nco"),
                                           ("cf32", "Z", "freqshift")])
def test_wideband_receiver_value_classes(rfm, port, synth, fmt, cls, mixer):
    """WidebandReceiver end to end (baseband, audio, RDS bits, status) against OracleStation / OracleNcoStation on
    the converted samples, two calls."""
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    from oracle.wideband import OracleStation
    from oracle.wideband_nco import OracleNcoStation
    from test_gpu_iq_formats import _oracle_baseband
    n_call = BLK * BPC
    u8 = synth.make_wideband_u8(FS, 2 * n_call, FREQS)
    x = requantise(u8, fmt, seed=2)
    raw = {"R +6 dB clipped": lambda: requantise(u8, fmt, seed=2, gain=2.0), "M 2^-100": lambda: scaled(x, -100),
           "Z": lambda: with_zero_runs(x, BLK, 1)}[cls]()
    wb = wb_mod.WidebandReceiver(torch, FREQS, FS, BLK, BPC, mixer=mixer, device=0, input_format=fmt)
    oracles = [OracleNcoStation(f, FS, BLK, BPC) if mixer == "nco" else OracleStation(f, FS, BLK, BPC, mixer=mixer)
               for f in FREQS]
    for k in range(2):
        seg = slice(k * n_call, (k + 1) * n_call)
        audio = wb.process_iq(raw[seg])
        bb = wb.bb.cpu().numpy()
        conv = to_cf32(raw[seg])
        for s, o in enumerate(oracles):
            ref_bb = o.baseband_cf32(conv) if mixer == "nco" else _oracle_baseband(o, conv)
            assert nan_equal(bb[s], ref_bb), (fmt, cls, mixer, k, s, "baseband")
            assert nan_equal(audio[s], o.dec.process_cf32(ref_bb)), (fmt, cls, mixer, k, s, "audio")
    for s, o in enumerate(oracles):
        assert np.array_equal(wb.dec.take_bits(s), o.dec.take_bits())
        assert _same_status(wb.dec.status(s), o.dec.status())
        o.close()
    wb.close()


# ---------------------------------------------------------------------------------------------------------------------
# band scan
# ---------------------------------------------------------------------------------------------------------------------
FS_RTL, N_CALL_RTL = 2.4e6, 128000
RASTER_RTL = (-1.1e6, 100e3, 23)
SCAN_N = 2 * N_CALL_RTL


@pytest.fixture(scope="module")
def rtl_u8(synth):
    return synth.make_wideband_u8(FS_RTL, SCAN_N, [-800e3, 300e3])


def _scan_classes(u8):
    out = {}
    for fmt in ("s8", "s16", "cf32"):
        x = requantise(u8, fmt, seed=4)
        out[f"{fmt} Z"] = with_zero_runs(x, 65536, 1)
        if fmt == "cf32":
            for k in M_EXPONENTS:
                out[f"cf32 M 2^{k}"] = scaled(x, k)
        else:
            out[f"{fmt} R"] = with_rails(x, 65536)
            out[f"{fmt} R +6 dB clipped"] = requantise(u8, fmt, seed=4, gain=2.0)
    return out


# |X|^2 of a 4096-point Hann segment reaches about (2^k * 2048)^2: float32 overflows from k = 53 (2^61 and above are
# refused), and below k = -64 every bin underflows in the float32 partial sums (the spectrum is zero, not wrong)
def _scan_regime(name: str) -> str:
    if " M " not in name:
        return "compare"
    k = int(name.split("2^")[1])
    return "refused" if k >= 53 else ("compare" if k >= -64 else "underflow")


def test_scan_value_classes(rfm, rtl_u8):
    """Spectrum against oracle/scan.py's float64 Welch spectrum within the existing tolerance relative to the total
    power, and channel powers and candidates the restatement's bit for bit, for Z, R and M inside the float32 range;
    M beyond it is refused."""
    for name, cap in _scan_classes(rtl_u8).items():
        s = rfm.BandScan(FS_RTL, *RASTER_RTL, device=0)
        regime = _scan_regime(name)
        if regime == "refused":
            with pytest.raises(rfm.RadioFmError, match="not finite"):
                s.run(cap)
            s.close()
            continue
        s.run(cap)
        psd, chan, st = s.spectrum(), s.channel_power(), s.stations()
        assert np.all(np.isfinite(psd)) and np.all(psd >= 0), name
        bins = scan.channel_bins(FS_RTL, *RASTER_RTL)
        assert np.array_equal(chan.view(np.uint64), scan.channel_powers(psd, bins).view(np.uint64)), name
        assert [d["freq"] for d in st] == [RASTER_RTL[0] + j * RASTER_RTL[1] for j in scan.candidates(chan)], name
        if regime == "compare":
            ref = welch_psd_iq(cap)
            tot = float(ref.sum())
            assert float(np.max(np.abs(psd.astype(np.float64) - ref))) <= 1e-6 * tot, name
        s.close()


def _scan_result(s):
    return s.spectrum(), s.channel_power(), s.stations(), s.iq_correction()


@pytest.mark.filterwarnings("ignore::RuntimeWarning")          # the float64 restatement of a NaN capture
@pytest.mark.parametrize("mode", ["off", "fixed", "estimate"])
def test_scan_refuses_a_non_finite_spectrum(rfm, rtl_u8, mode):
    """A NaN sample, an Inf sample and a finite 1e30 capture (whose float32 spectrum overflows) make rfm_scan_run
    return RFM_ERR_INVALID with the reason, before any decision; BandScan raises RadioFmError.  The same handle then
    gives, for a clean capture, what a fresh handle gives."""
    corr = {"off": None, "fixed": rfm.IqCorrection(0.01, -0.02, 1.05, 0.03), "estimate": "estimate"}[mode]
    clean = requantise(rtl_u8, "cf32")
    nan, inf, big = clean.copy(), clean.copy(), (clean.astype(np.float64) * 1e30).astype(np.float32)
    nan[70000, 0] = np.nan
    inf[70001, 1] = np.inf
    assert np.all(np.isfinite(big))
    s = rfm.BandScan(FS_RTL, *RASTER_RTL, device=0, iq_correction=corr)
    for label, cap in (("nan", nan), ("inf", inf), ("1e30", big)):
        with pytest.raises(rfm.RadioFmError, match="not finite"):
            s.run(cap)
        with pytest.raises(rfm.RadioFmError):
            s.spectrum()                                 # no completed run
        with pytest.raises(ValueError):                  # the restatement applies the same rule
            scan.channel_powers(welch_psd_iq(cap).astype(np.float32), scan.channel_bins(FS_RTL, *RASTER_RTL))
    s.run(clean)
    a = _scan_result(s)
    s.close()
    f = rfm.BandScan(FS_RTL, *RASTER_RTL, device=0, iq_correction=corr)
    f.run(clean)
    b = _scan_result(f)
    f.close()
    assert bits_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
    assert a[2] == b[2] and a[3] == b[3] and len(a[2]) >= 2, (a[2], b[2])


# ---------------------------------------------------------------------------------------------------------------------
# IQ estimate
# ---------------------------------------------------------------------------------------------------------------------
def _est_tuple(c):
    return (np.float32(c.dc_i), np.float32(c.dc_q), np.float32(c.a), np.float32(c.b), bool(c.imbalance_valid))


def test_iq_estimate_value_classes(rfm):
    """cf32 at the M scales against the float64 restatement (1e-12), all-zero and constant-rail captures, and
    non-finite cf32: a non-finite dc, a = 1, b = 0, imbalance_valid = 0 (host and device input alike)."""
    torch = _torch()
    rng = np.random.default_rng(6)
    n = 3 * 16384 + 5
    x = (rng.standard_normal((n, 2)) * 0.3 + [0.01, -0.02]).astype(np.float32)
    x[:, 1] = (0.9 * x[:, 1] + 0.1 * x[:, 0]).astype(np.float32)
    for k in M_EXPONENTS:
        cap = scaled(x, k)
        host = rfm.estimate_iq_correction(cap)
        dev = rfm.estimate_iq_correction(torch.from_numpy(cap).cuda())
        assert dev == host, k
        ref = iqcorr.coefficients_float64(cap)
        for nm, got, r in zip(("dc_i", "dc_q", "a", "b"), _est_tuple(host)[:4], ref[:4]):
            lo, hi = sorted((float(r) * (1 - 1e-12), float(r) * (1 + 1e-12)))
            assert np.float32(lo) <= got <= np.float32(hi), (k, nm, got, r)
        assert host.imbalance_valid == ref[4], k
    for dt, v in ((np.int8, 0), (np.int16, 0), (np.float32, 0.0), (np.int8, -128), (np.int16, -32768),
                  (np.int8, 127), (np.int16, 32767)):
        cap = np.full((n, 2), v, dtype=dt)
        got = _est_tuple(rfm.estimate_iq_correction(cap))
        want = iqcorr.estimate(cap)
        assert got == tuple(want[:4]) + (bool(want[4]),), (dt, v, got, want)
        assert got[2:] == (1.0, 0.0, False)
    for bad in (np.nan, np.inf, -np.inf):
        cap = x.copy()
        cap[1000, 1] = bad
        for c in (rfm.estimate_iq_correction(cap), rfm.estimate_iq_correction(torch.from_numpy(cap).cuda())):
            assert not np.isfinite(c.dc_q) and c.a == 1.0 and c.b == 0.0 and not c.imbalance_valid, (bad, c)


ESTIMATE_LIMIT = 1 << 32


@pytest.mark.parametrize("fmt,pattern", [("s8", "rail"), ("s16", "rail"), ("s8", "alternating")])
def test_iq_estimate_at_its_stated_limit(rfm, fmt, pattern):
    """n = 2^32 samples on the device (8 GiB of s8, 16 GiB of s16), bit for bit against the closed-form integer sums;
    n = 2^32 + 1 is refused."""
    torch = _torch()
    dt, esz, lo, hi = {"s8": (torch.int8, 2, -128, 127), "s16": (torch.int16, 4, -32768, 32767)}[fmt]
    need = (ESTIMATE_LIMIT + 1) * esz
    free, _ = torch.cuda.mem_get_info(0)
    if free < need + (1 << 30):
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    n = ESTIMATE_LIMIT
    cap = torch.empty((n + 1, 2), dtype=dt, device="cuda")
    if pattern == "rail":
        cap.fill_(lo)
        i_codes, q_codes = (lo, lo), (lo, lo)
    else:                                    # I: lo, hi, lo, ...; Q: hi, lo, hi, ...
        cap[0::2, 0] = lo
        cap[1::2, 0] = hi
        cap[0::2, 1] = hi
        cap[1::2, 1] = lo
        i_codes, q_codes = (lo, hi), (hi, lo)
    torch.cuda.synchronize()
    h = n // 2
    si, sq = h * sum(i_codes), h * sum(q_codes)
    sii, sqq = h * sum(v * v for v in i_codes), h * sum(v * v for v in q_codes)
    siq = h * sum(a * b for a, b in zip(i_codes, q_codes))
    want = iqcorr.coefficients_from_integer_sums(iqcorr.S8 if fmt == "s8" else iqcorr.S16, (n, si, sq, sii, sqq, siq))
    got = rfm.estimate_iq_correction(cap.data_ptr(), fmt=fmt, n=n, device=0)
    assert _est_tuple(got) == tuple(want[:4]) + (bool(want[4]),), (fmt, pattern, got, want)
    with pytest.raises(rfm.RadioFmError):
        rfm.estimate_iq_correction(cap.data_ptr(), fmt=fmt, n=n + 1, device=0)
    del cap
    torch.cuda.empty_cache()
