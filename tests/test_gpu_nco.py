"""Phase-accumulator NCO on the device (rfm_downconvert_set_nco, WidebandReceiver(mixer="nco"), rfm_scan_set_mixer).

The NCO is exact float32 arithmetic on a phase the project defines (oracle/nco.py), in front of paths that are pinned
to the reference elsewhere.  So a down-converter with the NCO set must give, bit for bit, what the same object gives
without it for cf32 rows of the host-mixed samples, and the "nco" receiver and scan must equal
OracleNcoStation (oracle/wideband_nco.py).  The audible check at the end is why the mixer exists: the freqshift table's 1562.5 Hz
buzz on a station 9.8 MHz from the centre, which the NCO does not have."""
import importlib
import subprocess

import numpy as np
import pytest

from conftest import bits_equal
from oracle import iqcorr, nco
from test_iq_formats import to_cf32
from test_nco import build_nco_driver

pytestmark = pytest.mark.gpu

RFM_ERR_INVALID = -1
FMTS = ["u8", "s8", "s16", "cf32"]
FS, BLK, BPC = 50.0e6, 32000, 64
N_CALL = BLK * BPC
RASTER_50M = (-24.9e6, 100e3, 499)


def _torch():
    import torch
    return torch


def _raw(u8: np.ndarray, fmt: str, seed: int = 0) -> np.ndarray:
    """The u8 capture in container fmt: s8 = u - 128, s16 = 256 (u - 128) + a random low byte, cf32 = the conversion."""
    if fmt == "u8":
        return u8
    if fmt == "cf32":
        return to_cf32(u8)
    v = u8.astype(np.int32) - 128
    if fmt == "s8":
        return v.astype(np.int8)
    return (v * 256 + np.random.default_rng(seed).integers(0, 256, size=v.shape)).astype(np.int16)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the down-converter: NCO set == host-mixed cf32 rows, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
PLANS = {   # label -> (fs, max_bw, wfm, call lengths in units of 2^stages)
    "wfm50M": (50.0e6, 100000.0, True, (5000, 1000, 9000, 2000)),           # uniform kernel, 7 x HB51, time chunks
    "wfm2.4M": (2.4e6, 100000.0, True, (6000, 1000, 12000, 500)),            # uniform kernel, 3 x HB51
    "generic2.4M": (2.4e6, 100000.0, False, (3000, 500, 6000, 250)),         # generic kernel (SetDataRate)
}


def _nco_freqs(fs):
    # a station, an off-raster station and the Nyquist edge (the word 2^31); -f brings +f to 0 Hz
    return np.array([-0.196 * fs, -3_333_317.3 * fs / 50.0e6, -fs / 2])


@pytest.fixture(scope="module")
def nco_u8(synth):
    return synth.make_wideband_u8(50.0e6, 17000 * 128, [9.8e6, 3_333_317.3, 200000.0])


@pytest.mark.parametrize("corr", [False, True])
@pytest.mark.parametrize("plan", list(PLANS))
@pytest.mark.parametrize("fmt", FMTS)
def test_downconvert_with_nco_equals_host_mixed_cf32_rows(rfm, nco_u8, fmt, plan, corr):
    torch = _torch()
    fs, bw, wfm, units = PLANS[plan]
    probe = rfm.DownConvertBatch([0.0], fs, bw, wfm=wfm, max_len=4096, device=0)
    nst = probe.n_stages
    assert (probe.stage_taps == [51] * nst) == wfm
    probe.close()
    lengths = [u << nst for u in units]
    total = sum(lengths)
    raw = _raw(nco_u8[:total], fmt)
    conv = to_cf32(raw)
    c = rfm.estimate_iq_correction(raw) if corr else None
    if corr:
        conv = iqcorr.apply(conv, c.dc_i, c.dc_q, c.a, c.b)
    rows = np.stack([raw, raw[::-1], np.roll(raw, 1000, axis=0)])
    rows_conv = np.stack([to_cf32(r) for r in rows])
    if corr:
        rows_conv = iqcorr.apply(rows_conv, c.dc_i, c.dc_q, c.a, c.b)
    f1 = _nco_freqs(fs)
    f2 = np.array([0.31 * fs, -1234.5, 0.0])      # set in the middle of the stream
    dev = torch.device("cuda", 0)
    mx = max(lengths)
    for shared in (True, False):
        dn = rfm.DownConvertBatch([0.0] * 3, fs, bw, wfm=wfm, max_len=mx, device=0)
        dr = rfm.DownConvertBatch([0.0] * 3, fs, bw, wfm=wfm, max_len=mx, device=0)
        if corr:
            dn.set_iq_correction(c)
        dn.set_nco(f1)
        host = [nco.Nco(f, np.float32(fs)) for f in f1]
        pos = 0
        for k, n in enumerate(lengths):
            if k == 2:      # re-set the NCO mid-stream: every phase restarts at 0, the filters carry on
                dn.set_nco(f2)
                host = [nco.Nco(f, np.float32(fs)) for f in f2]
            if k == 3:      # reset: filters, NCO_OSC and NCO phase
                dn.reset()
                dr.reset()
                for h in host:
                    h.reset()
            seg = slice(pos, pos + n)
            pos += n
            src = [conv[seg]] * 3 if shared else [rows_conv[r, seg] for r in range(3)]
            mixed = np.ascontiguousarray(np.stack([h.mix(x) for h, x in zip(host, src)]))
            m = n >> nst
            if shared and k % 2 == 0:      # device entry point
                x = torch.from_numpy(np.ascontiguousarray(raw[seg])).to(dev)
                out = torch.empty((3, m, 2), dtype=torch.float32, device=dev)
                assert dn.process_iq_device(fmt, True, x.data_ptr(), 0, out.data_ptr(), m, n) == m
                torch.cuda.synchronize()
                got = out.cpu().numpy()
            else:
                got = dn.process_iq(raw[seg] if shared else np.ascontiguousarray(rows[:, seg]), shared_capture=shared)
            want = dr.process_cf32(mixed)
            assert bits_equal(got, want), (fmt, plan, corr, shared, k)
            assert float(np.max(np.abs(want))) > 1e-3
        dn.close()
        dr.close()


def test_nco_off_equals_an_object_that_never_had_it(rfm, nco_u8):
    fs, n = 50.0e6, 8000 * 128
    x = to_cf32(nco_u8[:2 * n])
    a = rfm.DownConvertBatch([0.0, 1.0e6], fs, 100000.0, wfm=True, max_len=n, device=0)
    b = rfm.DownConvertBatch([0.0, 1.0e6], fs, 100000.0, wfm=True, max_len=n, device=0)
    f = np.array([-9.8e6, 2.5e6])
    a.set_nco(f)
    mixed = np.stack([nco.mix(x[:n], v, np.float32(fs)) for v in f])
    assert bits_equal(a.process_iq(x[:n], shared_capture=True), b.process_cf32(mixed))
    a.set_nco(None)
    assert bits_equal(a.process_iq(x[n:], shared_capture=True), b.process_iq(x[n:], shared_capture=True))
    a.reset()
    b.reset()
    assert bits_equal(a.process_iq(x[:n], shared_capture=True), b.process_iq(x[:n], shared_capture=True))
    a.close()
    b.close()


def test_argument_errors(rfm):
    L = rfm.lib()
    fs = 2.4e6
    dc = rfm.DownConvertBatch([0.0, 0.0], fs, 100000.0, max_len=4096, device=0)
    half = float(np.float32(fs)) / 2
    for bad in ([np.nextafter(half, np.inf), 0.0], [0.0, -np.nextafter(half, np.inf)], [np.nan, 0.0], [0.0, np.inf]):
        with pytest.raises(rfm.RadioFmError):
            dc.set_nco(bad)
        assert b"in_rate" in L.rfm_last_error()
    dc.set_nco([half, -half])                     # the edges themselves are allowed
    with pytest.raises(ValueError):
        dc.set_nco([0.0])
    torch = _torch()
    tab = torch.zeros((2, 64, 2), dtype=torch.float32, device="cuda")
    with pytest.raises(rfm.RadioFmError):        # one pre-mixer at a time
        dc.set_premix(tab.data_ptr(), 64, 64)
    dc.set_nco(None)
    dc.set_premix(tab.data_ptr(), 64, 64)
    with pytest.raises(rfm.RadioFmError):
        dc.set_nco([0.0, 0.0])
    dc.set_premix(0, 0, 0)
    dc.set_nco([0.0, 0.0])
    dc.close()
    s = rfm.BandScan(fs, -1.1e6, 100e3, 23, device=0)
    for m in (-1, 2):
        assert L.rfm_scan_set_mixer(s._h, m) == RFM_ERR_INVALID
        assert b"mixer" in L.rfm_last_error()
    assert L.rfm_scan_set_mixer(s._h, 1) == 0 and L.rfm_scan_set_mixer(s._h, 0) == 0
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. WidebandReceiver(mixer="nco") against OracleNcoStation
# ---------------------------------------------------------------------------------------------------------------------
EDGE_FREQS = [-24.9e6, 0.0, 3_333_317.3, 24.9e6]   # band edges, centre, and an off-raster station


@pytest.mark.parametrize("fmt", ["u8", "s16"])
def test_wideband_receiver_nco_equals_the_oracle(rfm, port, synth, fmt):
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    from oracle.wideband_nco import OracleNcoStation
    with pytest.raises(AssertionError, match="phase-coherent"):   # what freqshift makes of the off-raster station
        wb_mod.WidebandReceiver(torch, EDGE_FREQS, FS, BLK, BPC, mixer="freqshift", device=0)
    u8 = synth.make_wideband_u8(FS, 2 * N_CALL, EDGE_FREQS)
    raw = _raw(u8, fmt)
    conv = to_cf32(raw)
    wb = wb_mod.WidebandReceiver(torch, EDGE_FREQS, FS, BLK, BPC, mixer="nco", device=0, input_format=fmt)
    oracles = [OracleNcoStation(f, FS, BLK, BPC) for f in EDGE_FREQS]
    peak = 0.0
    for k in range(2):
        sl = slice(k * N_CALL, (k + 1) * N_CALL)
        audio = wb.process_iq(raw[sl])
        bb = wb.bb.cpu().numpy()
        for s, o in enumerate(oracles):
            ref_bb = o.baseband_cf32(conv[sl])
            assert bits_equal(bb[s], ref_bb), (fmt, k, s, "baseband")
            ref_audio = o.dec.process_cf32(ref_bb)
            assert bits_equal(audio[s], ref_audio), (fmt, k, s, "audio")
            peak = max(peak, float(np.max(np.abs(ref_audio))))
    assert peak > 0.02
    for s, o in enumerate(oracles):
        assert np.array_equal(wb.dec.take_bits(s), o.dec.take_bits()), s
        so, sd = o.dec.status(), wb.dec.status(s)
        assert all(np.float32(so[k]) == np.float32(sd[k]) for k in so), (s, so, sd)
        o.close()
    wb.close()


def _pi_ps(rfm, groups):
    vals, first, cnt = np.unique(groups[:, 0], return_index=True, return_counts=True)
    best = max(range(len(vals)), key=lambda i: (cnt[i], -first[i]))
    g = rfm.RdsGroupDecoder()
    g.decode(groups)
    ps = g.channel_name().rstrip(b"\0").decode("latin-1")
    g.close()
    return int(vals[best]), ps


@pytest.fixture(scope="module")
def c5_capture():
    """The scan's C5 second: 100 stations on the 200 kHz raster, 24 calls (0.98 s), made on the device."""
    torch = _torch()
    sd = importlib.import_module("radiofm_b200.synth_device")
    freqs = [(k - 50) * 200000.0 for k in range(100)]
    cap = sd.make_wideband_u8(torch, FS, 24 * N_CALL, freqs, torch.device("cuda", 0))
    torch.cuda.synchronize()
    return freqs, cap


def test_wideband_receiver_nco_100_stations(rfm, synth, c5_capture):
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    freqs, cap = c5_capture
    wb = wb_mod.WidebandReceiver(torch, freqs, FS, BLK, BPC, mixer="nco", device=0)
    for c in range(24):
        wb.process_device(cap.data_ptr() + 2 * c * N_CALL)
    wb.wait()
    torch.cuda.synchronize()
    for s in range(100):
        p = synth.stream_params(s % 4)
        assert wb.dec.status(s)["stereo"], s
        pi, ps = _pi_ps(rfm, wb.dec.take_groups(s))
        assert pi == p["pi"] and ps == p["ps"], (s, hex(pi), ps)
    wb.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. the scan with mixer="nco"
# ---------------------------------------------------------------------------------------------------------------------
def _scan(rfm, cap, mixer, **kw):
    s = rfm.BandScan(FS, *RASTER_50M, device=0, mixer=mixer, **kw)
    s.run(cap)
    st = s.stations()
    t = s.timing()
    s.close()
    return st, t


def test_scan_nco_on_the_c5_second(rfm, port, synth, c5_capture):
    from oracle.wideband_nco import OracleNcoStation
    freqs, cap = c5_capture
    st_osc, t_osc = _scan(rfm, cap, "osc")
    st, t = _scan(rfm, cap, "nco")
    print(f"[scan nco] confirmation {t[1]:.1f} ms (osc {t_osc[1]:.1f} ms), spectrum {t[0]:.3f} ms")
    assert [d["freq"] for d in st] == [d["freq"] for d in st_osc] == freqs
    for k, d in enumerate(st):
        p = synth.stream_params(k % 4)
        assert d["stereo"] and d["pi"] == p["pi"] and d["ps"] == p["ps"], (k, d)
    host = cap.cpu().numpy()
    st_host, _ = _scan(rfm, host, "nco")
    assert st_host == st
    for k in (0, 50, 99):
        o = OracleNcoStation(freqs[k], FS, BLK, BPC)
        for c in range(24):
            o.process_u8(host[c * N_CALL:(c + 1) * N_CALL])
        so, groups = o.dec.status(), o.dec.take_groups()
        d = st[k]
        assert d["stereo"] == bool(so["stereo"])
        for a in ("pilot_level", "if_level", "bb_level"):
            assert bits_equal(np.atleast_1d(d[a]), np.atleast_1d(np.float32(so[a]))), (k, a)
        assert d["rds_groups"] == len(groups) > 0
        assert (d["pi"], d["ps"]) == _pi_ps(rfm, groups), k
        o.close()
    # with the IQ correction estimated per run
    st_e, _ = _scan(rfm, cap, "nco", iq_correction="estimate")
    assert [d["freq"] for d in st_e] == freqs
    for k, d in enumerate(st_e):
        p = synth.stream_params(k % 4)
        assert d["stereo"] and d["pi"] == p["pi"] and d["ps"] == p["ps"], (k, d)


# ---------------------------------------------------------------------------------------------------------------------
# 4. the audible check: the freqshift table's 1562.5 Hz buzz at +9.8 MHz, and its absence with the NCO
# ---------------------------------------------------------------------------------------------------------------------
F_TONE_STATION = 9.8e6     # 9.8e6 * 32000 / 50e6 = 6272: phase-coherent, so freqshift accepts it
CALLS_AUDIBLE = 26         # the first two are left out: 0.98 s of settled audio


def _tone_station_cs16(call: int) -> np.ndarray:
    """One call of a mono FM station at +9.8 MHz carrying a 1 kHz tone at half deviation, -6 dBFS, in white noise 30 dB
    below it over the 50 MHz band (54 dB in a 200 kHz channel): the noise gives the audio a floor to measure against."""
    i = np.arange(call * N_CALL, (call + 1) * N_CALL, dtype=np.float64)
    ph = 2.0 * np.pi * ((F_TONE_STATION * i) % FS) / FS + 37.5 * np.sin(2.0 * np.pi * 1000.0 * i / FS)
    z = 0.5 * np.exp(1j * ph)
    w = np.random.default_rng(call).standard_normal((N_CALL, 2)) * (0.5 * 10 ** (-30 / 20) / np.sqrt(2))
    x = np.stack([z.real, z.imag], axis=1) + w
    return np.clip(np.rint(32768.0 * x), -32768, 32767).astype(np.int16)


def _audio(wb_mod, torch, mixer, calls):
    wb = wb_mod.WidebandReceiver(torch, [F_TONE_STATION], FS, BLK, BPC, mixer=mixer, device=0, input_format="s16")
    out = [wb.process_iq(c)[0].copy() for c in calls]
    wb.close()
    return np.concatenate(out[2:])[0::2].astype(np.float64)     # left channel, settled


def _buzz_levels(left: np.ndarray, fs_audio: float = 48000.0):
    """Welch power (Blackman-Harris, 2048 points: 23.4 Hz bins, about 45 averages) at k x 1562.5 Hz (k = 1..5), the
    largest of the three nearest bins, over the median of the bins 7 to 16 bins away on either side, in dB."""
    from scipy.signal import welch
    hz_axis, p = welch(left, fs=fs_audio, window="blackmanharris", nperseg=2048, noverlap=1024)
    hz = hz_axis[1]
    out = []
    for k in range(1, 6):
        j = int(round(k * 1562.5 / hz))
        nb = np.concatenate([p[j - 16:j - 6], p[j + 7:j + 17]])
        out.append(10 * np.log10(np.max(p[j - 1:j + 2]) / np.median(nb)))
    return out


def test_freqshift_buzz_and_the_nco(rfm):
    torch = _torch()
    wb_mod = importlib.import_module("radiofm_b200.wideband")
    calls = [_tone_station_cs16(c) for c in range(CALLS_AUDIBLE)]
    lv = {m: _buzz_levels(_audio(wb_mod, torch, m, calls)) for m in ("freqshift", "nco")}
    for m, v in lv.items():
        print(f"[nco audible] {m}: k x 1562.5 Hz (k = 1..5) over the neighbouring median: "
              + ", ".join(f"{x:+.1f}" for x in v) + " dB")
    assert max(lv["nco"]) <= 3.0, lv["nco"]
    assert min(lv["freqshift"]) >= 20.0, lv["freqshift"]


# ---------------------------------------------------------------------------------------------------------------------
# 5. the C++ driver: an "nco" scan and a down-converter with the NCO, C ABI only
# ---------------------------------------------------------------------------------------------------------------------
RTL_STATIONS = [(-800e3, 11), (-300e3, 12), (200e3, 13)]
FS_RTL = 2.4e6


def test_nco_driver_scans_and_decodes(rfm, synth, tmp_path):
    n = int(FS_RTL)
    acc = np.zeros(n, dtype=np.complex128)
    for f, sid in RTL_STATIONS:
        p = synth.stream_params(sid)
        bits = synth.rds_bits_from_groups(synth.rds_group_stream(p["pi"], p["ps"], 16))
        mpx = synth.mpx_signal(FS_RTL, n, left=p["left"], right=p["right"], pilot=0.1, rds_level=0.05, rds_bits=bits)
        acc += (1.0 if f != -300e3 else 0.7) * np.exp(
            1j * (2.0 * np.pi * 75000.0 / FS_RTL * np.cumsum(mpx) + 2.0 * np.pi * f * np.arange(n) / FS_RTL))
    acc *= 0.8 / float(np.max(np.abs(acc)))
    cap = np.clip(np.rint(127.5 + 127.5 * np.stack([acc.real, acc.imag], axis=1)), 0, 255).astype(np.uint8)
    cap.tofile(tmp_path / "cap.u8")
    exe = build_nco_driver(tmp_path)
    out = subprocess.run([exe, str(tmp_path / "cap.u8"), str(FS_RTL), "-1.1e6", "100e3", "23"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    print(out.stdout)
    assert "scan: 3 stations" in out.stdout and "refusals: ok" in out.stdout
    s = rfm.BandScan(FS_RTL, -1.1e6, 100e3, 23, device=0, mixer="nco")
    s.run(cap)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("station:")]
    for ln, d in zip(lines, s.stations()):
        assert ln.startswith(f"station: offset_hz={d['freq']:.0f} ") and f"pi={d['pi']:X} ps={d['ps']}" in ln, ln
    s.close()
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("decoded:")][0]
    head, ps = line.split(" ps=", 1)
    fields = dict(kv.split("=", 1) for kv in head.split()[1:])
    p = synth.stream_params(dict(RTL_STATIONS)[float(fields["offset_hz"])])
    assert fields["stereo"] == "1" and int(fields["groups"]) > 0 and fields["pi"] == f"{p['pi']:X}" and ps == p["ps"]
