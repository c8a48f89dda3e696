"""IQ correction on the device (rfm_iq_estimate, *_set_iq_correction, the scan's modes).

The estimate must be oracle/iqcorr.py's (bit for bit for the integer formats), and a corrected run must give, bit for
bit, what the same object gives for cf32 rows of the host-corrected samples (oracle/iqcorr.apply) with no correction:
the correction is exact float32 arithmetic in front of paths that are pinned elsewhere."""
import ctypes as C
import importlib
import subprocess

import numpy as np
import pytest

from conftest import bits_equal
from oracle import iqcorr, scan
from test_gpu_iq_formats import _oracle_baseband
from test_iq_correction import build_iqcorr_driver, imbalanced, quantise
from test_iq_formats import to_cf32, welch_psd_iq

pytestmark = pytest.mark.gpu

RFM_ERR_INVALID = -1
FMTS = ["u8", "s8", "s16", "cf32"]


def _torch():
    import torch
    return torch


def _capture(fmt: str, n: int, seed: int = 0) -> np.ndarray:
    """A proper noise-like signal with 1 dB / 3 degrees of imbalance and a DC offset, in container fmt ([n, 2])."""
    rng = np.random.default_rng(seed)
    z = 0.25 * (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2)
    return quantise(imbalanced(z, 1.0, 3.0, dc=(0.02, 0.015)), fmt)


def _corr(rfm, c) -> "object":
    return rfm.IqCorrection(*c[:4], bool(c[4]))


def _apply(cap, c) -> np.ndarray:
    return iqcorr.apply(to_cf32(cap), c.dc_i, c.dc_q, c.a, c.b)


# ---------------------------------------------------------------------------------------------------------------------
# 1. estimator
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["u8", "s8", "s16"])
def test_integer_estimate_is_bit_identical_to_the_restatement(rfm, fmt):
    torch = _torch()
    # odd, shorter than one CTA's 16384 samples, a few CTAs with a partial last one, many CTAs
    for n in (1, 1001, 5 * 16384 + 77, 2_400_000):
        cap = _capture(fmt, n, seed=n)
        want = _corr(rfm, iqcorr.estimate(cap))
        host = rfm.estimate_iq_correction(cap)
        d = torch.from_numpy(np.ascontiguousarray(cap)).cuda()
        torch.cuda.synchronize()
        dev, again = rfm.estimate_iq_correction(d), rfm.estimate_iq_correction(d)
        assert host == want and dev == want and again == want, (fmt, n, host, want)
        assert (n == 1) != want.imbalance_valid


def test_cf32_estimate_agrees_with_the_float64_restatement(rfm):
    torch = _torch()
    for n in (1001, 5 * 16384 + 77, 2_400_000):
        cap = _capture("cf32", n, seed=n)
        host = rfm.estimate_iq_correction(cap)
        d = torch.from_numpy(cap).cuda()
        torch.cuda.synchronize()
        dev = rfm.estimate_iq_correction(d)
        assert dev == host and rfm.estimate_iq_correction(d) == host, n
        ref = iqcorr.coefficients_float64(cap)
        # the device value is the float rounding of a double within 1e-12 relative of the exactly summed one
        for name, got, r in zip(("dc_i", "dc_q", "a", "b"), (host.dc_i, host.dc_q, host.a, host.b), ref[:4]):
            lo, hi = sorted((float(r) * (1 - 1e-12), float(r) * (1 + 1e-12)))
            assert np.float32(lo) <= got <= np.float32(hi), (n, name, got, r)
        assert host.imbalance_valid


# ---------------------------------------------------------------------------------------------------------------------
# 2. application: corrected input == uncorrected cf32 rows of the host-corrected samples, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
PLANS = {   # label -> (fs, max_bw, wfm, n, nco): a uniform HB51 chain and a mixed generic one
    "wfm50M": (50.0e6, 100000.0, True, 2 * 32000 * 64 // 2, [-1.0e6, 200000.0, 7.0e6]),
    "generic2.4M": (2.4e6, 100000.0, False, 65536, [-300000.0, 0.0, 500000.0]),
}


@pytest.fixture(scope="module")
def corr_u8(synth):
    return synth.make_wideband_u8(50.0e6, 32000 * 64, [-1.0e6, 200000.0, 7.0e6])


def _raw(u8, fmt, n, seed=0):
    """The wideband u8 capture requantised to fmt, with imbalance added in float64 (a zero-IF receiver's view)."""
    x = to_cf32(u8[:n]).astype(np.float64)
    z = x[:, 0] + 1j * x[:, 1]
    return quantise(0.9 * imbalanced(z, 1.0, 3.0, dc=(0.02, 0.015)) / 1.1, fmt)


@pytest.mark.parametrize("premix", [False, True])
@pytest.mark.parametrize("plan", list(PLANS))
@pytest.mark.parametrize("fmt", FMTS)
def test_downconvert_with_correction_equals_corrected_cf32_rows(rfm, corr_u8, fmt, plan, premix):
    torch = _torch()
    fs, bw, wfm, n, nco = PLANS[plan]
    raw = _raw(corr_u8, fmt, n)
    c = rfm.estimate_iq_correction(raw)
    assert c.imbalance_valid
    fixed = _apply(raw, c)
    rows = np.stack([raw, raw[::-1], np.roll(raw, 1000, axis=0)])
    rows_fixed = np.stack([_apply(r, c) for r in rows])
    dev = torch.device("cuda", 0)
    tab = None
    if premix:
        ph = 4000
        fsb = rfm.FreqShiftBatch([-f for f in nco], fs, max_len=ph, device=0)
        ones = np.zeros((3, ph, 2), dtype=np.float32)
        ones[:, :, 0] = 1.0
        tab = torch.from_numpy(fsb.process_cf32(ones)).to(dev)
        fsb.close()
    outs = {}
    for label in ("shared corrected", "shared reference", "rows corrected", "rows reference"):
        dc = rfm.DownConvertBatch(nco if not premix else [0.0] * 3, fs, bw, wfm=wfm, max_len=n, device=0)
        if premix:
            dc.set_premix(tab.data_ptr(), tab.shape[1], tab.shape[1])
        m = n >> dc.n_stages
        out = torch.empty((3, m, 2), dtype=torch.float32, device=dev)
        if label == "shared corrected":
            dc.set_iq_correction(c)
            x = torch.from_numpy(np.ascontiguousarray(raw)).to(dev)
            k = dc.process_iq_device(fmt, True, x.data_ptr(), 0, out.data_ptr(), m, n)
        elif label == "shared reference":
            x = torch.from_numpy(fixed).to(dev)
            k = dc.process_iq_device("cf32", False, x.data_ptr(), 0, out.data_ptr(), m, n)
        elif label == "rows corrected":
            dc.set_iq_correction(c)
            x = torch.from_numpy(np.ascontiguousarray(rows)).to(dev)
            k = dc.process_iq_device(fmt, False, x.data_ptr(), n, out.data_ptr(), m, n)
        else:
            x = torch.from_numpy(rows_fixed).to(dev)
            k = dc.process_iq_device("cf32", False, x.data_ptr(), n, out.data_ptr(), m, n)
        torch.cuda.synchronize()
        assert k == m
        outs[label] = out.cpu().numpy()
        if label == "shared corrected":   # the host entry point, same object state after a reset
            dc.reset()
            if premix:
                dc.set_premix(tab.data_ptr(), tab.shape[1], tab.shape[1])
            outs["shared corrected host"] = dc.process_iq(raw, shared_capture=True)
            dc.set_iq_correction(None)     # off again: the plain conversion
            dc.reset()
            if premix:
                dc.set_premix(tab.data_ptr(), tab.shape[1], tab.shape[1])
            outs["shared uncorrected"] = dc.process_iq(raw, shared_capture=True)
        dc.close()
    assert bits_equal(outs["shared corrected"], outs["shared reference"]), (fmt, plan, premix)
    assert bits_equal(outs["shared corrected host"], outs["shared reference"]), (fmt, plan, premix)
    assert bits_equal(outs["rows corrected"], outs["rows reference"]), (fmt, plan, premix)
    assert not bits_equal(outs["shared uncorrected"], outs["shared reference"])
    assert float(np.max(np.abs(outs["shared reference"]))) > 1e-3


@pytest.mark.parametrize("fmt", FMTS)
def test_freqshift_with_correction_equals_corrected_cf32_rows(rfm, corr_u8, fmt):
    n = 40000
    raw = _raw(corr_u8, fmt, n)
    c = rfm.estimate_iq_correction(raw)
    nco = [-1.0e6, 0.0, 7.0e6]
    a, b = (rfm.FreqShiftBatch(nco, 50.0e6, max_len=n, device=0) for _ in range(2))
    a.set_iq_correction(c)
    got = a.process_iq(raw, shared_capture=True)
    want = b.process_cf32(np.stack([_apply(raw, c)] * 3))
    assert bits_equal(got, want), fmt
    a.reset()
    b.reset()
    rows = np.stack([raw, raw[::-1], raw])
    assert bits_equal(a.process_iq(rows, shared_capture=False), b.process_cf32(np.stack([_apply(r, c) for r in rows])))
    a.close()
    b.close()


@pytest.mark.parametrize("mixer", ["osc", "freqshift", "freqshift_unfused"])
@pytest.mark.parametrize("fmt", ["s8", "s16"])
def test_wideband_receiver_with_correction(rfm, port, synth, fmt, mixer):
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    from oracle.wideband import OracleStation
    FS, BLK, BPC, FREQS = 50.0e6, 32000, 64, [-1.0e6, 200000.0, 7.0e6]
    n_call = BLK * BPC
    u8 = synth.make_wideband_u8(FS, 2 * n_call, FREQS)
    raw = _raw(u8, fmt, 2 * n_call)
    c = rfm.estimate_iq_correction(raw)
    fixed = _apply(raw, c)
    wb = wb_mod.WidebandReceiver(torch, FREQS, FS, BLK, BPC, mixer=mixer, device=0, input_format=fmt, iq_correction=c)
    oracles = [OracleStation(f, FS, BLK, BPC, mixer=mixer.split("_")[0]) for f in FREQS]
    for k in range(2):
        sl = slice(k * n_call, (k + 1) * n_call)
        audio = wb.process_iq(raw[sl])
        bb = wb.bb.cpu().numpy()
        for s, o in enumerate(oracles):
            ref_bb = _oracle_baseband(o, fixed[sl])
            assert bits_equal(bb[s], ref_bb), (fmt, mixer, k, s, "baseband")
            assert bits_equal(audio[s], o.dec.process_cf32(ref_bb)), (fmt, mixer, k, s, "audio")
    for s, o in enumerate(oracles):
        assert np.array_equal(wb.dec.take_bits(s), o.dec.take_bits())
        o.close()
    wb.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. scan
# ---------------------------------------------------------------------------------------------------------------------
FS_RTL = 2.4e6
RASTER = (-1.1e6, 100e3, 23)
GHOST = [(300e3, 41), (-600e3, 42), (900e3, 43)]   # (offset, synth stream id); mirrors 200 kHz from any station


def _fm(mpx, fs, f):
    return np.exp(1j * (2.0 * np.pi * 75000.0 / fs * np.cumsum(mpx) + 2.0 * np.pi * f * np.arange(mpx.size) / fs))


@pytest.fixture(scope="module")
def ghost_window(synth):
    """A HackRF-like 2.4 MS/s zero-IF window: three stereo RDS stations of equal power with free mirror channels,
    1 dB / 3 degrees of IQ imbalance and a DC offset of (0.02, 0.015), modulated in float64 and quantised once to
    cs8 and to u8."""
    n = int(FS_RTL)
    acc = np.zeros(n, dtype=np.complex128)
    for f, sid in GHOST:
        p = synth.stream_params(sid)
        bits = synth.rds_bits_from_groups(synth.rds_group_stream(p["pi"], p["ps"], 16))
        mpx = synth.mpx_signal(FS_RTL, n, left=p["left"], right=p["right"], pilot=0.1, rds_level=0.05, rds_bits=bits)
        acc += _fm(mpx, FS_RTL, f)
    acc *= 0.85 / float(np.max(np.abs(acc)))
    x = imbalanced(acc, 1.0, 3.0, dc=(0.02, 0.015))
    return quantise(x, "s8"), quantise(x, "u8")


def test_scan_fixed_correction_spectrum_channels_and_stations(rfm, ghost_window):
    cap = ghost_window[0]
    c = rfm.estimate_iq_correction(cap)
    s = rfm.BandScan(FS_RTL, *RASTER, device=0, iq_correction=c)
    s.run(cap)
    assert s.iq_correction() == c
    psd, chan, st = s.spectrum(), s.channel_power(), s.stations()
    ref = welch_psd_iq(_apply(cap, c))
    tot = float(ref.sum())
    assert float(np.max(np.abs(psd.astype(np.float64) - ref))) <= 1e-6 * tot
    bins = scan.channel_bins(FS_RTL, *RASTER)
    c_ref = scan.channel_powers(ref, bins)
    sel = c_ref >= scan.noise_floor(c_ref)
    assert float(np.max(np.abs(scan.channel_powers(psd, bins)[sel] - c_ref[sel]) / c_ref[sel])) <= 1e-4
    assert np.array_equal(chan.view(np.uint64), scan.channel_powers(psd, bins).view(np.uint64))
    assert [d["freq"] for d in st] == [RASTER[0] + j * RASTER[1] for j in scan.candidates(chan)]
    # mode 1 applies exactly what rfm_iq_estimate gives, host and device input alike
    torch = _torch()
    s2 = rfm.BandScan(FS_RTL, *RASTER, device=0, iq_correction="estimate")
    s2.run(cap)
    assert s2.iq_correction() == c
    assert bits_equal(s2.spectrum(), psd) and s2.stations() == st
    d = torch.from_numpy(np.ascontiguousarray(cap)).cuda()
    torch.cuda.synchronize()
    s2.run(d)
    assert s2.iq_correction() == c and bits_equal(s2.spectrum(), psd)
    # off again: the plain spectrum, and the identity reported
    s2.set_iq_correction(None)
    s2.run(cap)
    assert s2.iq_correction() == rfm.IqCorrection(0.0, 0.0, 1.0, 0.0, False)
    assert float(np.max(np.abs(s2.spectrum().astype(np.float64) - welch_psd_iq(cap)))) <= 1e-6 * tot
    s.close()
    s2.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. why: the ghosts of a zero-IF capture
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["s8", "u8"])
def test_mirror_ghosts_and_dc_disappear_with_the_estimate(rfm, synth, ghost_window, fmt):
    cap = ghost_window[0 if fmt == "s8" else 1]
    j = lambda f: int(round((f - RASTER[0]) / RASTER[1]))
    s = rfm.BandScan(FS_RTL, *RASTER, device=0)
    s.run(cap)
    st0 = {d["freq"]: d for d in s.stations()}
    chan0 = s.channel_power()
    for f, sid in GHOST:
        assert -f in st0, (fmt, -f, sorted(st0))
        g = st0[-f]
        print(f"[ghost] {fmt} mirror of {f / 1e3:+.0f} kHz: {10 * np.log10(chan0[j(f)] / chan0[j(-f)]):.1f} dB below, "
              f"stereo {g['stereo']}, {g['rds_groups']} RDS groups, PI {g['pi']:#x}, PS {g['ps']!r}")
        if g["rds_groups"]:
            assert g["pi"] == synth.stream_params(sid)["pi"], (fmt, f, g)
    assert 0.0 in st0, (fmt, sorted(st0))
    s.set_iq_correction("estimate")
    s.run(cap)
    st = {d["freq"]: d for d in s.stations()}
    chan = s.channel_power()
    assert sorted(st) == sorted(f for f, _ in GHOST), (fmt, sorted(st))
    for f, sid in GHOST:
        rej = 10 * np.log10(chan[j(f)] / chan[j(-f)])
        print(f"[ghost] {fmt} corrected: station {f / 1e3:+.0f} kHz {rej:.1f} dB over its mirror")
        assert rej >= 45.0, (fmt, f, rej)
        p = synth.stream_params(sid)
        assert st[f]["stereo"] and st[f]["pi"] == p["pi"] and st[f]["ps"] == p["ps"], (fmt, st[f])
    print(f"[ghost] {fmt} corrected: 0 Hz channel {10 * np.log10(chan[j(0.0)] / chan[j(GHOST[0][0])]):.1f} dB "
          f"below a station; estimate {s.iq_correction()}")
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. argument errors
# ---------------------------------------------------------------------------------------------------------------------
def test_argument_errors(rfm):
    torch = _torch()
    L = rfm.lib()
    s = rfm.BandScan(FS_RTL, *RASTER, device=0)
    for mode in (-1, 3):
        assert L.rfm_scan_set_iq_correction(s._h, mode, None) == RFM_ERR_INVALID
        assert b"mode" in L.rfm_last_error()
    assert L.rfm_scan_set_iq_correction(s._h, 2, None) == RFM_ERR_INVALID
    assert b"NULL" in L.rfm_last_error()
    bad = rfm.RfmIqCorrection(float("nan"), 0.0, 1.0, 0.0, 1)
    assert L.rfm_scan_set_iq_correction(s._h, 2, C.byref(bad)) == RFM_ERR_INVALID
    d = torch.zeros((4096, 2), dtype=torch.int16, device="cuda")
    out = rfm.RfmIqCorrection()
    assert L.rfm_iq_estimate(rfm.IQ_S16, C.c_void_p(d.data_ptr() + 2), 4000, 1, 0, C.byref(out)) == RFM_ERR_INVALID
    assert b"aligned" in L.rfm_last_error()
    # the binding refuses what it cannot map to a mode before calling the library
    with pytest.raises(ValueError):
        s.set_iq_correction("estimated")
    with pytest.raises(TypeError):
        s.set_iq_correction((0.0, 0.0, 1.0, 0.0))
    # the mode-1 scan refuses the misaligned capture with the same reason
    s.set_iq_correction("estimate")
    big = torch.zeros((int(FS_RTL) + 8, 2), dtype=torch.int16, device="cuda")
    assert L.rfm_scan_run(s._h, rfm.IQ_S16, C.c_void_p(big.data_ptr() + 2), int(FS_RTL), 1) == RFM_ERR_INVALID
    assert b"aligned" in L.rfm_last_error()
    dc = rfm.DownConvertBatch([0.0], 2.4e6, 100000.0, max_len=4096, device=0)
    assert L.rfm_downconvert_set_iq_correction(dc._h, C.byref(bad)) == RFM_ERR_INVALID
    fsb = rfm.FreqShiftBatch([0.0], 2.4e6, max_len=4096, device=0)
    assert L.rfm_freqshift_set_iq_correction(fsb._h, C.byref(bad)) == RFM_ERR_INVALID
    s.close()
    dc.close()
    fsb.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. the C++ driver: estimate -> scan with the estimate -> decode one station, C ABI only
# ---------------------------------------------------------------------------------------------------------------------
def test_iqcorr_driver_estimates_scans_and_decodes(rfm, synth, ghost_window, tmp_path):
    exe = build_iqcorr_driver(tmp_path)
    cap = ghost_window[0]
    cap.tofile(tmp_path / "cap.cs8")
    out = subprocess.run([exe, str(tmp_path / "cap.cs8"), str(FS_RTL), *[str(v) for v in RASTER]],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    print(out.stdout)
    c = rfm.estimate_iq_correction(cap)
    est = dict(kv.split("=") for kv in out.stdout.splitlines()[0].split()[1:])
    assert np.float32(est["a"]) == c.a and np.float32(est["b"]) == c.b and np.float32(est["dc_i"]) == c.dc_i
    assert "scan: 3 stations, applied same" in out.stdout
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("decoded:")][0]
    head, ps = line.split(" ps=", 1)
    fields = dict(kv.split("=", 1) for kv in head.split()[1:])
    sid = dict(GHOST)[float(fields["offset_hz"])]
    p = synth.stream_params(sid)
    assert fields["stereo"] == "1" and int(fields["groups"]) > 0 and fields["pi"] == f"{p['pi']:X}"
    assert ps == p["ps"]
