"""Pin the oracle: the plain-C restatement (oracle/radiofm_oracle.c) against
  (1) the UNMODIFIED reference compiled in place (oracle/_ref/libradiofm_ref.so) -- bit for bit on every
      stage tap, audio, status, RDS bits and groups, at all BASELINE.json rates;
  (2) the committed golden fixtures (tests/golden/*.npz) that were generated from that reference library
      (tests/golden/make_golden.py) -- so the pin also holds where the reference library is absent.
The reference ships no tests or golden vectors (SURVEY.md section 4).  CPU only.
"""
import ctypes as C
import functools
import hashlib
import os
import sys

import numpy as np
import pytest

from conftest import RATES, bits_equal, station

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
f32p = C.POINTER(C.c_float)
P = lambda a: a.ctypes.data_as(f32p)


# ---------------------------------------------------------------------------------------------------
# (1) against the compiled reference
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate,nblk", [("1.0M", 10), ("1.2M", 4), ("2.4M", 4), ("390k", 6)])
def test_port_matches_reference_every_stage(port, ref, rate, nblk):
    fs, ds, blk = RATES[rate]
    iq, _ = station(rate, nblk)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    r = ref.RefFmDecoder(fs, -0.15 * fs, downsample=ds)
    assert np.array_equal(o.constants()[:51], r.constants()[:51])
    for w in range(6):
        assert bits_equal(o.table(w), r.table(w)), f"table {w}"
    for b in range(nblk):
        x8 = iq[b * blk:(b + 1) * blk]
        x = ref.u8_to_cf32(x8)
        assert bits_equal(x, port.u8_to_cf32(x8))
        a_r, t_r = r.process_staged(x)
        a_o = o.process_u8(x8)
        assert bits_equal(a_o, a_r), f"audio block {b}"
        t_o = o.taps()
        for name in ref.TAP_NAMES:
            assert bits_equal(t_o[name], t_r[name]), f"tap {name} block {b}"
        assert t_o["stereo"] == t_r["stereo"]
        so, sr = o.status(), r.status()
        assert all(np.float32(so[k]) == np.float32(sr[k]) for k in so), (so, sr)
    assert np.array_equal(o.take_groups(), r.take_groups())
    assert np.array_equal(o.take_bits(), r.take_bits())


def test_port_reset_matches_reference(port, ref):
    fs, ds, blk = RATES["1.0M"]
    iq, _ = station("1.0M", 4)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    r = ref.RefFmDecoder(fs, -0.15 * fs, downsample=ds)
    for b in (0, 1):
        assert bits_equal(o.process_u8(iq[b * blk:(b + 1) * blk]), r.process_u8(iq[b * blk:(b + 1) * blk]))
    o.reset(); r.reset()
    for b in (2, 3):
        assert bits_equal(o.process_u8(iq[b * blk:(b + 1) * blk]), r.process_u8(iq[b * blk:(b + 1) * blk]))
    assert np.array_equal(o.take_groups(), r.take_groups())


def test_port_noisy_and_mono_match_reference(port, ref, synth):
    fs, ds, blk = RATES["1.0M"]
    for kw in ({"snr_db": 25.0, "stream_id": 3}, {"mono_tone": (1000.0, 0.5)}, {"stereo": False, "rds": False}):
        iq, _ = synth.make_station_u8(fs, 3 * blk, **kw)
        o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
        r = ref.RefFmDecoder(fs, -0.15 * fs, downsample=ds)
        for b in range(3):
            assert bits_equal(o.process_u8(iq[b * blk:(b + 1) * blk]), r.process_u8(iq[b * blk:(b + 1) * blk])), kw


def test_port_atan2f_is_libm_atan2f(port):
    """The restated glibc atan2f against the libm the reference links (same image on the GPU box)."""
    libm = C.CDLL("libm.so.6")
    libm.atan2f.restype = C.c_float
    libm.atan2f.argtypes = [C.c_float, C.c_float]
    rng = np.random.default_rng(5)
    n = 200_000
    y = np.concatenate([rng.standard_normal(n), rng.standard_normal(n) * 1e-3, rng.standard_normal(n)]).astype(np.float32)
    x = np.concatenate([rng.standard_normal(n), rng.standard_normal(n), rng.standard_normal(n) * 1e-4]).astype(np.float32)
    f, g = port.lib().rfo_atan2f, libm.atan2f
    bad = sum(1 for a, b in zip(y.tolist(), x.tolist()) if np.float32(f(a, b)).view(np.uint32) != np.float32(g(a, b)).view(np.uint32))
    assert bad == 0
    for a, b in ((0.0, 1.0), (0.0, -1.0), (-0.0, -1.0), (1.0, 0.0), (-1.0, 0.0), (1.0, 1.0), (1e30, 1e-30), (1e-30, -1e30)):
        assert np.float32(f(a, b)).view(np.uint32) == np.float32(g(a, b)).view(np.uint32), (a, b)


def test_port_sincos_is_rounded_double(port):
    rng = np.random.default_rng(6)
    ph = (rng.random(100_000) * 7.0 - 0.3).astype(np.float32)
    s, c = C.c_float(), C.c_float()
    for p in ph[:20000].tolist():
        port.lib().rfo_sincos(p, C.byref(s), C.byref(c))
        assert np.float32(s.value) == np.float32(np.sin(np.float64(p))) and np.float32(c.value) == np.float32(np.cos(np.float64(p)))


# ---------------------------------------------------------------------------------------------------
# (2) against the committed golden fixtures (generated from the reference library)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate", ["1.0M", "1.2M", "2.4M", "390k"])
def test_port_matches_golden_chain(port, rate):
    g = np.load(os.path.join(GOLDEN, f"chain_{rate}.npz"))
    fs, ds, n = float(g["fs"]), int(g["ds"]), int(g["n"])
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    assert np.array_equal(o.constants()[:51], g["constants"][:51])
    for w in range(6):
        assert bits_equal(o.table(w), g[f"table{w}"])
    lut = port.u8_to_cf32(np.arange(256, dtype=np.uint8).repeat(2).reshape(-1, 2))[:, 0]
    assert bits_equal(lut, g["cf32_first"])
    for k in range(3):
        a = o.process_u8(g["iq"][k * n:(k + 1) * n])
        assert bits_equal(a, g[f"audio{k}"]), f"audio call {k}"
        assert bits_equal(np.array([float(v) for v in o.status().values()], dtype=np.float32), g[f"status{k}"])
    t = o.taps()
    for name in port.TAP_NAMES:
        if name != "tuned":
            assert bits_equal(t[name], g["tap_" + name]), name


def test_port_matches_golden_rds(port):
    g = np.load(os.path.join(GOLDEN, "rds_1.0M.npz"))
    fs, ds, blk, nblk = float(g["fs"]), int(g["ds"]), int(g["blk"]), int(g["nblk"])
    iq, sent = station("1.0M", nblk)
    assert hashlib.sha256(iq.tobytes()).hexdigest() == str(g["iq_sha256"]), \
        "synthetic generator no longer reproduces the fixture's input bytes"
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    h = hashlib.sha256()
    for b in range(nblk):
        a = o.process_u8(iq[b * blk:(b + 1) * blk])
        h.update(a.tobytes())
        assert a.size == g["audio_len"][b] and o.status()["stereo"] == bool(g["stereo"][b])
    assert h.hexdigest() == str(g["audio_sha256"])
    groups = o.take_groups()
    assert np.array_equal(groups, g["groups"]) and np.array_equal(o.take_bits(), g["bits"])
    # the decoded groups are the transmitted ones, in order (SURVEY.md section 8c)
    assert len(groups) >= 3
    first = next(i for i in range(len(sent)) if np.array_equal(sent[i], groups[0]))
    assert np.array_equal(groups, sent[first:first + len(groups)])


def test_port_matches_golden_rds_block_kat(port):
    k = np.load(os.path.join(GOLDEN, "kat_rds_blocks.npz"))
    c = C.c_uint32(0)
    f = port.lib().rfo_rds_check_block
    for w, osyn, fec, syn, fixed in zip(k["word"].tolist(), k["offset_syndrome"].tolist(), k["use_fec"].tolist(),
                                        k["syndrome"].tolist(), k["corrected"].tolist()):
        assert f(w, osyn, fec, C.byref(c)) == syn and c.value == fixed


def test_fir_designs_match_golden(port):
    """cFirFilter::InitLPFilter / InitHPFilter taps (FirFilter.cpp:78-148, 195-264) of the C restatement and of the
    library's host-only planner entry point against the compiled reference's (three Kaiser-beta ranges, forced and
    clamped tap counts)."""
    from conftest import load_package
    rfm = load_package()
    g = np.load(os.path.join(GOLDEN, "kat_primitives.npz"))
    L = port.lib()
    off = 0
    for row, nt in zip(g["fir_design_specs"], g["fir_design_lens"].tolist()):
        kind, spec = int(row[0]), (int(row[1]),) + tuple(float(np.float32(v)) for v in row[2:])
        want = g["fir_design_taps"][off:off + nt]
        off += nt
        h = L.rfo_fir_create()
        assert (L.rfo_fir_init_hp if kind else L.rfo_fir_init_lp)(h, *spec) == nt, (kind, spec)
        co = np.zeros(160, dtype=np.float32)
        L.rfo_fir_coef(h, P(co))
        L.rfo_fir_destroy(h)
        assert bits_equal(co[:nt], want), ("port", kind, spec)
        assert bits_equal(rfm.fir_design("hp" if kind else "lp", *spec), want), ("library", kind, spec)
    assert off == g["fir_design_taps"].size


def test_port_matches_golden_primitives(port):
    g = np.load(os.path.join(GOLDEN, "kat_primitives.npz"))
    L = port.lib()
    # cFreqShift
    h = L.rfo_freqshift_create(37000.0, 1.0e6)
    y = g["freqshift_in"].copy()
    L.rfo_freqshift_process(h, P(y), 1500)
    L.rfo_freqshift_process(h, P(y[1500:]), 1500)
    L.rfo_freqshift_destroy(h)
    assert bits_equal(y, g["freqshift_out"])
    x = g["freqshift_in"]
    # cDownsampleFilter integer (complex)
    h = L.rfo_downsample_create(32, 0.15, 4.0, 1)
    y = np.zeros((3000, 2), dtype=np.float32)
    k1 = L.rfo_downsample_process_complex(h, P(x), P(y), 1501)
    k2 = L.rfo_downsample_process_complex(h, P(x[1501:]), P(y[k1:]), 1499)
    L.rfo_downsample_destroy(h)
    assert [k1, k2] == g["ds_int_split"].tolist() and bits_equal(y[:k1 + k2], g["ds_int_out"])
    # fractional (real)
    r = np.ascontiguousarray(x[:, 0])
    h = L.rfo_downsample_create(250, 15000.0 / 250000.0, 250000.0 / 48000.0, 0)
    y = np.zeros(3000, dtype=np.float32)
    k1 = L.rfo_downsample_process_real(h, P(r), P(y), 1700)
    k2 = L.rfo_downsample_process_real(h, P(r[1700:]), P(y[k1:]), 1300)
    L.rfo_downsample_destroy(h)
    assert [k1, k2] == g["ds_frac_split"].tolist() and bits_equal(y[:k1 + k2], g["ds_frac_out"])
    # integer (real), the last call shorter than the filter order
    h = L.rfo_downsample_create(40, 0.12, 5.0, 1)
    y = np.zeros(3000, dtype=np.float32)
    k1 = L.rfo_downsample_process_real(h, P(r), P(y), 1501)
    k2 = L.rfo_downsample_process_real(h, P(r[1501:]), P(y[k1:]), 1478)
    k3 = L.rfo_downsample_process_real(h, P(r[2979:]), P(y[k1 + k2:]), 21)
    L.rfo_downsample_destroy(h)
    assert [k1, k2, k3] == g["ds_rint_split"].tolist() and bits_equal(y[:k1 + k2 + k3], g["ds_rint_out"])
    # CRDSDownConvert
    h = L.rfo_rdsdc_create()
    L.rfo_rdsdc_set_frequency(h, -57000.0)
    rate = L.rfo_rdsdc_set_data_rate(h, 250000.0, 4800.0)
    lens = (C.c_int * 16)()
    ns = L.rfo_rdsdc_stages(h, lens, 16)
    z = g["rdsdc_in"].copy()
    y = np.zeros((2048, 2), dtype=np.float32)
    k1 = L.rfo_rdsdc_process(h, 1024, P(z), P(y))
    k2 = L.rfo_rdsdc_process(h, 1024, P(z[1024:]), P(y[k1:]))
    L.rfo_rdsdc_destroy(h)
    assert np.float32(rate) == g["rdsdc_rate"] and list(lens[:ns]) == g["rdsdc_stages"].tolist()
    assert bits_equal(y[:k1 + k2], g["rdsdc_out"])
    # cFirFilter
    h = L.rfo_fir_create()
    nt = L.rfo_fir_init_lp(h, 0, 1.0, 60.0, 15000.0, 21000.0, 48000.0)
    co = np.zeros(80, dtype=np.float32)
    L.rfo_fir_coef(h, P(co))
    a, b = np.ascontiguousarray(x[:1000, 0]), np.ascontiguousarray(x[:1000, 1])
    L.rfo_fir_process_two(h, P(a), P(b), 1000)
    L.rfo_fir_destroy(h)
    assert bits_equal(co[:nt], g["fir_lp_taps"]) and bits_equal(a, g["fir_two_a"]) and bits_equal(b, g["fir_two_b"])
    # cIirFilter
    for name, typ, f0, q, fs in (("notch", 3, 19000.0, 5.0, 48000.0), ("bp", 2, 1187.5, 500.0, 31250.0)):
        h = L.rfo_iir_create()
        L.rfo_iir_init(h, typ, f0, q, fs)
        co = np.zeros(5, dtype=np.float32)
        L.rfo_iir_coef(h, P(co))
        a = np.ascontiguousarray(x[:1000, 0])
        L.rfo_iir_process_real(h, P(a), 1000)
        L.rfo_iir_destroy(h)
        assert bits_equal(co, g[f"iir_{name}_coef"]) and bits_equal(a, g[f"iir_{name}_out"]), name
    # cPilotPhaseLock
    pil = g["pilot_in"]
    n = pil.size
    h = L.rfo_pilot_create(np.float32(19000.0 / 250000.0), np.float32(50.0 / 250000.0), np.float32(0.04))
    y = np.zeros(n, dtype=np.float32)
    l1 = L.rfo_pilot_process(h, P(pil), P(y), n // 2)
    l2 = L.rfo_pilot_process(h, P(pil[n // 2:]), P(y[n // 2:]), n // 2)
    lvl = L.rfo_pilot_level(h)
    L.rfo_pilot_destroy(h)
    assert bits_equal(y, g["pilot_out"]) and [l1, l2] == g["pilot_lock"].tolist() and np.float32(lvl) == g["pilot_level"]


@pytest.mark.parametrize("in_rate,max_bw,wfm,freq,n", [
    (4.0e6, 4800.0, False, 100000.0, 16384),      # CIC3, fixed 11-tap x4, HB15, HB23, HB47
    (2.4e6, 100000.0, False, -57000.0, 8192),     # HB15, HB23, HB51
    (50.0e6, 100000.0, True, -7.0e6, 32000),      # SetWfmDataRate: 7 x HB51
    (50.0e6, 100000.0, True, 0.0, 12800),         # 0 Hz: the oscillator falls into its 4-cycle
])
def test_rdsdc_port_vs_ref_every_stage_kind(port, ref, in_rate, max_bw, wfm, freq, n):
    """The C restatement of CRDSDownConvert against the compiled reference for the stage kinds and planners the decoder's
    own RDS chain never exercises (they back the stand-alone rfm_downconvert primitive and the wideband front end)."""
    rng = np.random.default_rng(11)
    LP, LR = port.lib(), ref.lib()
    hp, hr = LP.rfo_rdsdc_create(), LR.ref_rdsdc_create()
    LP.rfo_rdsdc_set_frequency(hp, np.float32(freq))
    LR.ref_rdsdc_set_frequency(hr, np.float32(freq))
    if wfm:
        rp = LP.rfo_rdsdc_set_wfm_data_rate(hp, np.float32(in_rate), np.float32(max_bw))
        rr = LR.ref_rdsdc_set_wfm_data_rate(hr, np.float32(in_rate), np.float32(max_bw))
    else:
        rp = LP.rfo_rdsdc_set_data_rate(hp, np.float32(in_rate), np.float32(max_bw))
        rr = LR.ref_rdsdc_set_data_rate(hr, np.float32(in_rate), np.float32(max_bw))
    assert np.float32(rp) == np.float32(rr)
    for _ in range(3):
        x = (rng.standard_normal((n, 2)) * 0.3).astype(np.float32)
        zp, zr = x.copy(), x.copy()
        yp, yr = np.zeros_like(x), np.zeros_like(x)
        kp = LP.rfo_rdsdc_process(hp, n, P(zp), P(yp))
        kr = LR.ref_rdsdc_process(hr, n, P(zr), P(yr))
        assert kp == kr and bits_equal(yp[:kp], yr[:kr])
    LP.rfo_rdsdc_destroy(hp)
    LR.ref_rdsdc_destroy(hr)


# ---------------------------------------------------------------------------------------------------
# (3) the cases of (1) against tests/golden/ref_cases.npz (tests/golden/make_golden_ref_cases.py): the same
#     comparisons where the original is not built
# ---------------------------------------------------------------------------------------------------
GOLD_REF = np.load(os.path.join(GOLDEN, "ref_cases.npz"))


@functools.lru_cache(maxsize=None)
def ref_cases(use_ref: bool) -> dict:
    sys.path.insert(0, GOLDEN)
    import make_golden_ref_cases as mr
    return mr.make(use_ref)


def same_as_golden(prefix: str):
    got = ref_cases(False)
    keys = [k for k in GOLD_REF.files if k.startswith(prefix)]
    assert keys
    for k in keys:
        assert np.array_equal(got[k], GOLD_REF[k]), k


@pytest.mark.parametrize("rate", ["1.0M", "1.2M", "2.4M", "390k"])
def test_port_matches_golden_every_stage(port, rate):
    same_as_golden(f"stage_{rate}_")


def test_port_reset_matches_golden(port):
    same_as_golden("reset_")


def test_port_noisy_and_mono_match_golden(port):
    same_as_golden("noisy_")


@pytest.mark.parametrize("j", range(4))
def test_rdsdc_port_matches_golden_every_stage_kind(port, j):
    same_as_golden(f"rdsdc{j}_")


def test_demux_port_packets_match_golden(port):
    """the restatement of cRadioReceiver::DemuxRead against the add-on's packets (test_ref_addon.py)"""
    same_as_golden("demux_")


def test_ref_cases_golden_is_what_the_reference_produces(port):
    sys.path.insert(0, GOLDEN)
    import make_golden_ref_cases as mr
    if not mr.reference_available():
        pytest.skip("oracle/_ref/ not built (see oracle/Makefile)")
    got = ref_cases(True)
    for k in GOLD_REF.files:
        if k != "source":
            assert np.array_equal(got[k], GOLD_REF[k]), k
