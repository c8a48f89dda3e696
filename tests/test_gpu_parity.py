"""Parity of the sm_100a chain against the oracle, through the C ABI (pytest -m gpu, on the B200 box).

Bars (BASELINE.json north_star): u8 conversion and RDS bits/groups bit-exact; audio within 1e-4 of full
scale max-abs; tone SNR within 0.1 dB.  The kernels restate the reference's arithmetic operation by
operation (rfm_math.cuh), so these tests assert the stronger property first -- every stage tap, the audio,
the level meters and the RDS bits are BIT-IDENTICAL to the oracle -- and then the north_star tolerances
explicitly (L+R and L-R separately, SURVEY.md section 0.5b).

The oracle used here is oracle/port.py (plain-C restatement, pinned bit-exact against the compiled reference
and the golden fixtures in tests/test_oracle_port.py); where oracle/_ref/libradiofm_ref.so travelled to the
box the unmodified reference is checked as well.
"""
import hashlib
import os
import sys

import numpy as np
import pytest

from conftest import RATES, ROOT, bits_equal, station

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLDEN)
GPU_TAPS = ["demod_in", "baseband", "rawstereo", "mono_rs", "stereo_rs", "lp_stereo", "lp_mono", "rds_dec",
            "rds_lp", "rds_pll", "rds_mf"]


def oracle_tap(o, name):
    if name in ("lp_stereo", "lp_mono"):
        full = o.tap("lp")
        na = full.size // 2
        return full[:na] if name == "lp_stereo" else full[na:]
    return o.tap(name)


def tolerances(a_gpu, a_ref):
    """north_star tolerances: audio <= 1e-4 max-abs; L+R <= 1e-6 and L-R <= 2e-4 separately."""
    assert a_gpu.shape == a_ref.shape
    if a_ref.size == 0:
        return
    assert float(np.max(np.abs(a_gpu - a_ref))) <= 1e-4
    g, r = a_gpu.reshape(-1, 2).astype(np.float64), a_ref.reshape(-1, 2).astype(np.float64)
    assert float(np.max(np.abs((g[:, 0] + g[:, 1]) - (r[:, 0] + r[:, 1])))) <= 1e-6
    assert float(np.max(np.abs((g[:, 0] - g[:, 1]) - (r[:, 0] - r[:, 1])))) <= 2e-4


# lanes_sms: 1 = no SM partition (what a single stream gets by default), 24 = the partition wide batches run in
# (rfm_config::lanes_sms: placement only -- the immediate-barrier lanes kernel and the persistent front end sized to the
# partition must produce the same bits)
@pytest.mark.parametrize("rate,nblk,lanes_sms", [("1.0M", 10, 1), ("1.2M", 11, 1), ("2.4M", 18, 1), ("390k", 12, 1),
                                                 ("2.4M", 18, 24), ("1.0M", 10, 16)])
def test_chain_every_stage_bit_exact(rfm, port, rate, nblk, lanes_sms):
    fs, ds, blk = RATES[rate]
    iq, sent = station(rate, nblk)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=1, max_block_len=blk, lanes_sms=lanes_sms)
    assert np.array_equal(o.constants()[:51], d.constants()[:51])
    saw_stereo = False
    for b in range(nblk):
        x = iq[b * blk:(b + 1) * blk]
        a_o = o.process_u8(x)
        a_d = d.process_u8(x[None])[0]
        tolerances(a_d, a_o)
        assert bits_equal(a_d, a_o), f"audio block {b}"
        for t in GPU_TAPS:
            assert bits_equal(d.tap(t), oracle_tap(o, t)), f"tap {t} block {b}"
        so, sd = o.status(), d.status()
        assert all(np.float32(so[k]) == np.float32(sd[k]) for k in so), (b, so, sd)
        saw_stereo |= sd["stereo"]
    assert saw_stereo, "window must cover the mono -> stereo switch-over"
    bits_o, bits_d = o.take_bits(), d.take_bits()
    assert bits_o.size > 50 and np.array_equal(bits_o, bits_d)
    g_o, g_d = o.take_groups(), d.take_groups()
    assert len(g_o) >= 2 and np.array_equal(g_o, g_d)
    first = next(i for i in range(len(sent)) if np.array_equal(sent[i], g_d[0]))
    assert np.array_equal(g_d, sent[first:first + len(g_d)]), "decoded groups are the transmitted ones, in order"


def test_against_unmodified_reference(rfm, ref):
    fs, ds, blk = RATES["1.2M"]
    iq, _ = station("1.2M", 11)
    r = ref.RefFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    for b in range(11):
        x = iq[b * blk:(b + 1) * blk]
        a_r, _ = r.process_staged(ref.u8_to_cf32(x), want=())
        a_d = d.process_u8(x[None])[0]
        tolerances(a_d, a_r)
        assert bits_equal(a_d, a_r)
    assert np.array_equal(r.take_bits(), d.take_bits()) and np.array_equal(r.take_groups(), d.take_groups())


def test_against_unmodified_reference_golden(rfm):
    """test_against_unmodified_reference's 11 blocks against the audio digests, bits and groups stored for them in
    tests/golden/ref_cases.npz (tests/golden/make_golden_ref_cases.py, checked against the original where it is built)."""
    from make_golden_ref_cases import sha
    g = np.load(os.path.join(GOLDEN, "ref_cases.npz"))
    fs, ds, blk = RATES["1.2M"]
    iq, _ = station("1.2M", 11)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    for b in range(11):
        assert sha(d.process_u8(iq[None, b * blk:(b + 1) * blk])[0]) == g["ref12_sha"][b], b
    assert np.array_equal(d.take_bits(), g["ref12_bits"]) and np.array_equal(d.take_groups(), g["ref12_groups"])


@pytest.mark.parametrize("rate", ["1.0M", "1.2M", "2.4M", "390k"])
def test_golden_chain_fixture(rfm, rate):
    g = np.load(os.path.join(GOLDEN, f"chain_{rate}.npz"))
    fs, ds, n = float(g["fs"]), int(g["ds"]), int(g["n"])
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=n)
    for k in range(3):
        a = d.process_u8(g["iq"][None, k * n:(k + 1) * n])[0]
        assert bits_equal(a, g[f"audio{k}"])
        assert bits_equal(np.array([float(v) for v in d.status().values()], dtype=np.float32), g[f"status{k}"])
    for t in ("demod_in", "baseband", "rawstereo", "mono_rs", "stereo_rs", "rds_dec", "rds_lp", "rds_pll", "rds_mf"):
        assert bits_equal(d.tap(t), g["tap_" + t]), t


def test_golden_rds_fixture(rfm):
    g = np.load(os.path.join(GOLDEN, "rds_1.0M.npz"))
    fs, ds, blk, nblk = float(g["fs"]), int(g["ds"]), int(g["blk"]), int(g["nblk"])
    iq, _ = station("1.0M", nblk)
    assert hashlib.sha256(iq.tobytes()).hexdigest() == str(g["iq_sha256"])
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    h = hashlib.sha256()
    for b in range(nblk):
        a = d.process_u8(iq[None, b * blk:(b + 1) * blk])[0]
        h.update(a.tobytes())
        assert a.size == g["audio_len"][b] and d.status()["stereo"] == bool(g["stereo"][b])
    assert h.hexdigest() == str(g["audio_sha256"])
    assert np.array_equal(d.take_groups(), g["groups"]) and np.array_equal(d.take_bits(), g["bits"])


def test_uecp_stream_of_the_batched_decoder(rfm):
    """SURVEY.md 8f N1 end to end: IQ -> ... -> groups -> per-stream cRDSGroupDecoder -> framed UECP bytes
    (rfm_decoder_rds_take_uecp), against the golden groups of the reference chain pushed through the oracle's
    restatement of the group decoder (itself pinned to the compiled reference in tests/test_uecp.py)."""
    from oracle import uecp_port
    g = np.load(os.path.join(GOLDEN, "rds_1.0M.npz"))
    fs, ds, blk, nblk = float(g["fs"]), int(g["ds"]), int(g["blk"]), int(g["nblk"])
    iq, _ = station("1.0M", nblk)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=2, max_block_len=blk)
    half = nblk // 2
    got = [b"", b""]
    for b in range(nblk):
        d.process_u8(np.stack([iq[b * blk:(b + 1) * blk]] * 2))
        if b == half:                     # draining in the middle must not lose or repeat a group
            got[0] += d.take_uecp(0)
            d.take_groups(0)
    for s in range(2):
        got[s] += d.take_uecp(s)
    o = uecp_port.OracleGroupDecoder()
    want = b"".join(uecp_port.stuff_frame(f) for f in o.decode(g["groups"]))
    assert len(g["groups"]) >= 4 and len(want) > 40
    assert got[0] == want and got[1] == want
    assert d.take_uecp(0) == b""


def test_reset_mid_stream_restarts_the_group_decoder(rfm, port):
    """cFmDecoder::Reset -> cRDSRxSignalProcessor::Reset -> cRDSGroupDecoder::Reset (RDSProcess.cpp:92,
    RDSGroupDecoder.cpp:140-164): after a reset on the same station the PI / PS / TA_TP / MS / DI frames are emitted
    again.  Oracle: the chain restatement (audio, groups, reset included) + the group-decoder restatement -- or the
    compiled reference group decoder where oracle/_ref travelled -- reset at the same block."""
    from oracle import uecp_port, ref_uecp
    fs, ds, blk = RATES["1.0M"]
    nblk, cut = 9, 7
    iq, _ = station("1.0M", nblk)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    decs = [uecp_port.OracleGroupDecoder()] + ([ref_uecp.RefGroupDecoder()] if ref_uecp.available() else [])
    want = [b"" for _ in decs]
    got = b""
    for rnd in range(2):
        for b in range(cut if rnd == 0 else nblk):
            x = iq[b * blk:(b + 1) * blk]
            assert bits_equal(d.process_u8(x[None])[0], o.process_u8(x)), (rnd, b)
        g = o.take_groups()
        assert len(g) >= 4 and np.array_equal(g, d.take_groups())
        for i, u in enumerate(decs):
            want[i] += b"".join(uecp_port.stuff_frame(f) for f in u.decode(g))
        got += d.take_uecp()
        if rnd == 0:
            d.reset(); o.reset()
            for u in decs:
                u.reset()
    assert all(w == got for w in want) and len(got) > 80
    # the PI frame (message element code 0x01) appears once per decoder life
    first = b"".join(uecp_port.stuff_frame(f) for f in uecp_port.OracleGroupDecoder().decode(g[:1]))
    assert got.count(first[:6]) >= 1


def test_two_devices_in_one_process(rfm, port):
    """per-device kernel attributes (dynamic shared memory limits) and state: a decoder on cuda:1 next to one on cuda:0"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (gpurun --gpus 2)")
    fs, ds, blk = RATES["2.4M"]
    iq, _ = station("2.4M", 2)
    outs = []
    for dev in (1, 0, 1):
        d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk, device=dev)
        outs.append([d.process_u8(iq[None, b * blk:(b + 1) * blk])[0] for b in range(2)])
        d.close()
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    want = [o.process_u8(iq[b * blk:(b + 1) * blk]) for b in range(2)]
    for got in outs:
        assert all(bits_equal(a, w) for a, w in zip(got, want))


def test_mono_tone_snr(rfm, port):
    """BASELINE config 0: 1 s of 1.0 MS/s, 1 kHz mono tone; SNR within 0.1 dB of the reference chain."""
    fs, ds, blk = RATES["1.0M"]
    iq, _ = station("1.0M", 15, mono=True)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    ao = np.concatenate([o.process_u8(iq[b * blk:(b + 1) * blk]) for b in range(15)])
    ad = np.concatenate([d.process_u8(iq[None, b * blk:(b + 1) * blk])[0] for b in range(15)])
    tolerances(ad, ao)

    def snr_db(a):
        x = a.reshape(-1, 2)[4800:, 0].astype(np.float64)
        t = np.arange(x.size) / 48000.0
        best = None
        for f in np.linspace(995.0, 1005.0, 41):
            A = np.stack([np.sin(2 * np.pi * f * t), np.cos(2 * np.pi * f * t), np.ones_like(t)], 1)
            c, *_ = np.linalg.lstsq(A, x, rcond=None)
            res = x - A @ c
            v = 10 * np.log10(np.sum((A[:, :2] @ c[:2]) ** 2) / np.sum(res ** 2))
            best = v if best is None or v > best else best
        return best

    s_o, s_d = snr_db(ao), snr_db(ad)
    assert s_o > 30.0 and abs(s_o - s_d) <= 0.1
    assert not d.status()["stereo"]


def test_batch_of_distinct_streams(rfm, port, synth):
    """Independent streams in one batch (incl. a noisy and a mono one) each equal their own oracle run; the
    stream-group pipelining (n_groups) must not change anything."""
    fs, ds, blk = RATES["2.4M"]
    S, nblk = 9, 3
    iqs, sents = [], []
    for s in range(S):
        kw = {"stream_id": s}
        if s == 4:
            kw["snr_db"] = 20.0
        if s == 7:
            kw.update(stereo=False, rds=False)
        iq, sent = synth.make_station_u8(fs, nblk * blk, **kw)
        iqs.append(iq)
    iqs = np.stack(iqs)
    ref_audio = []
    oracles = [port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds) for _ in range(S)]
    for b in range(nblk):
        ref_audio.append([oracles[s].process_u8(iqs[s, b * blk:(b + 1) * blk]) for s in range(S)])
    for n_groups in (1, 4):
        d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=S, max_block_len=blk, n_groups=n_groups)
        for b in range(nblk):
            a = d.process_u8(iqs[:, b * blk:(b + 1) * blk])
            for s in range(S):
                assert bits_equal(a[s], ref_audio[b][s]), (n_groups, b, s)
        for s in range(S):
            so, sd = oracles[s].status(), d.status(s)
            assert all(np.float32(so[k]) == np.float32(sd[k]) for k in so)
    for s in range(S):
        assert np.array_equal(oracles[s].take_bits(), d.take_bits(s))


def test_cf32_entry_point_and_reset(rfm, port):
    """ProcessStream(const ComplexType*, ...) signature (FmDecode.h:135) and Reset (FmDecode.cpp:326-338)."""
    fs, ds, blk = RATES["1.0M"]
    iq, _ = station("1.0M", 10)
    x = port.u8_to_cf32(iq).reshape(10, blk, 2)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    for b in range(4):
        assert bits_equal(d.process_cf32(x[b][None])[0], o.process_cf32(x[b]))
    o.reset(); d.reset()
    o.take_bits(); d.take_bits(); o.take_groups(); d.take_groups()
    for b in range(4, 10):
        assert bits_equal(d.process_cf32(x[b][None])[0], o.process_cf32(x[b])), b
        so, sd = o.status(), d.status()
        assert all(np.float32(so[k]) == np.float32(sd[k]) for k in so)
    assert np.array_equal(o.take_bits(), d.take_bits()) and np.array_equal(o.take_groups(), d.take_groups())


def test_ragged_block_lengths_and_edges(rfm, port):
    """Carried state across calls of different length (FIR tails, decimator phase, fractional resampler
    position, FIR rotation, PLL registers) -- the reference's caller may use any multiple of 4096."""
    fs, ds, blk = RATES["1.0M"]
    iq, _ = station("1.0M", 4)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk)
    pos = 0
    for n in (4096, 65536, 8192, 4128, 32768, 12320, 4096 * 7):
        x = iq[pos:pos + n]
        pos += n
        assert bits_equal(d.process_u8(x[None])[0], o.process_u8(x)), n
    assert np.array_equal(o.take_bits(), d.take_bits())
    # empty block: nothing written, no state change
    assert d.process_u8(np.zeros((1, 0, 2), dtype=np.uint8)).shape == (1, 0)
    x = iq[pos:pos + 4096]
    assert bits_equal(d.process_u8(x[None])[0], o.process_u8(x))
    # errors are reported, not swallowed
    with pytest.raises(rfm.RadioFmError, match="max_block_len"):
        d.process_u8(np.zeros((1, blk + 32, 2), dtype=np.uint8))
    with pytest.raises(rfm.RadioFmError, match="shorter than the input FIR order"):
        d.process_u8(np.zeros((1, 20, 2), dtype=np.uint8))
    import ctypes as C
    k = C.c_uint32(0)
    small = np.zeros(8, dtype=np.float32)
    rc = rfm.lib().rfm_decoder_process_u8(d._h, x.ctypes.data_as(C.POINTER(C.c_uint8)), 4096,
                                          small.ctypes.data_as(C.POINTER(C.c_float)), 8, C.byref(k))
    assert rc == -5  # RFM_ERR_OVERFLOW


def test_default_rtlsdr_block_at_1200k_and_odd_short_blocks(rfm, port):
    """Any block length yields audio, and the RDS branch follows the reference through the counts its half-band
    stages were not written for (DownConvert.cpp:498-550).  cRtlSdrSource's default block of 65536 samples at
    1.2 MS/s / 5 leaves 13107 or 13108 baseband samples: odd counts make (m + 1) / 2 outputs per stage and restart the
    decimation phase every block; blocks so short that a stage gets fewer samples than taps pass through unfiltered.
    Checked against the UNMODIFIED reference where oracle/_ref was built, and always against the oracle port and the
    per-block audio digests, bits and groups stored for these sizes in tests/golden/ref_cases.npz."""
    from make_golden_ref_cases import ODD_SIZES, sha
    from oracle import ref
    g = np.load(os.path.join(GOLDEN, "ref_cases.npz"))
    fs, ds = 1.2e6, 5
    blk = 65536
    iq, _ = station("1.2M", 12)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=2, max_block_len=blk)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    r = ref.RefFmDecoder(fs, -0.15 * fs, downsample=ds) if ref.available() else None
    pos = 0
    sizes = [blk] * 9 + [100, 333, 1000, 47, 4096, 65521, 777, 20000, 41, 65535, 4097]
    assert sizes == ODD_SIZES
    for i, n in enumerate(sizes):
        x = iq[pos:pos + n]
        pos += n
        a = d.process_u8(np.stack([x, x]))
        a_o = o.process_u8(x)
        assert sha(a_o) == g["odd_sha"][i], n
        if r is not None:
            a_r, _ = r.process_staged(ref.u8_to_cf32(x), want=())
            assert bits_equal(a_o, a_r), n
        assert bits_equal(a[0], a_o) and bits_equal(a[1], a_o), n
        assert bits_equal(d.tap("rds_dec"), o.tap("rds_dec")) and bits_equal(d.tap("rds_mf"), o.tap("rds_mf")), n
    bo = o.take_bits()
    assert bo.size > 700 and np.array_equal(bo, g["odd_bits"]) and (r is None or np.array_equal(bo, r.take_bits()))
    assert np.array_equal(d.take_bits(0), bo) and np.array_equal(d.take_bits(1), bo)
    go = o.take_groups()
    assert len(go) >= 5 and np.array_equal(go, g["odd_groups"]) and (r is None or np.array_equal(go, r.take_groups()))
    assert np.array_equal(d.take_groups(1), go)


@pytest.mark.parametrize("rate,n", [("2.4M", 65536), ("2.4M", 20000), ("1.2M", 4096), ("390k", 16004)])
def test_decimator_phase_walks_through_every_window_alignment(rfm, port, rate, n):
    """Block lengths that are not a multiple of the decimation make the decimator phase p0 -- and with it the first
    sample of every front-end window -- walk through all residues: the TMA boxes must start on 16-byte boundaries of
    global memory whatever p0 is (an odd 8-byte coordinate is an illegal instruction), the window is shifted by one
    slot for odd starts, rows whose pitch a tensor map cannot describe take the LDG kernel."""
    fs, ds, _ = RATES[rate]
    iq, _ = station(rate, 4)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=3, max_block_len=n)
    for b in range(min(12, iq.shape[0] // n)):
        x = iq[b * n:(b + 1) * n]
        a = d.process_u8(np.stack([x, x, x]))
        a_o = o.process_u8(x)
        assert bits_equal(a[0], a_o) and bits_equal(a[2], a_o), (rate, n, b)
        assert bits_equal(d.tap("demod_in", 1), o.tap("demod_in")), (rate, n, b)
    assert np.array_equal(d.take_bits(2), o.take_bits())


@pytest.mark.parametrize("rate,nblk", [("2.4M", 24), ("1.2M", 14)])
def test_tolerance_mode_stays_inside_the_north_star_tolerance(rfm, port, rate, nblk):
    """rfm_config::fir_fused = 1 (opt-in): fused multiply-adds in the front-end FIR, the resamplers and the rotating
    FIRs.  No longer bit-identical -- the test insists on that, so the switch cannot silently do nothing -- but inside
    BASELINE.json's tolerances against the oracle: audio 1e-4 of full scale, L+R 1e-6 x 10, L-R 2e-4, RDS bits and
    groups identical, same stereo decisions."""
    fs, ds, blk = RATES[rate]
    iq, _ = station(rate, nblk)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, max_block_len=blk, fir_fused=1)
    worst, exact = 0.0, True
    for b in range(nblk):
        x = iq[b * blk:(b + 1) * blk]
        a_o, a_d = o.process_u8(x), d.process_u8(x[None])[0]
        assert a_o.shape == a_d.shape
        worst = max(worst, float(np.max(np.abs(a_d - a_o))))
        exact &= bits_equal(a_d, a_o)
        g, r = a_d.reshape(-1, 2).astype(np.float64), a_o.reshape(-1, 2).astype(np.float64)
        assert float(np.max(np.abs((g[:, 0] + g[:, 1]) - (r[:, 0] + r[:, 1])))) <= 1e-5, b
        assert float(np.max(np.abs((g[:, 0] - g[:, 1]) - (r[:, 0] - r[:, 1])))) <= 2e-4, b
        assert d.status()["stereo"] == o.status()["stereo"], b
    assert 0.0 < worst <= 1e-4 and not exact, worst
    assert np.array_equal(d.take_bits(), o.take_bits()) and np.array_equal(d.take_groups(), o.take_groups())


def test_device_pointer_entry_point(rfm, port):
    """Device-resident IQ / audio on a caller-owned CUDA stream (what bench.py's `value` leg times)."""
    import torch
    fs, ds, blk = RATES["1.2M"]
    S = 5
    iq, _ = station("1.2M", 3)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=S, max_block_len=blk, n_groups=2)
    stride = d.max_audio_floats(blk)
    st = torch.cuda.Stream()
    for b in range(3):
        x = iq[b * blk:(b + 1) * blk]
        with torch.cuda.stream(st):
            t_in = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(x, (S,) + x.shape))).cuda(non_blocking=False)
            t_out = torch.zeros((S, stride), dtype=torch.float32, device="cuda")
            k = d.process_u8_device(t_in.data_ptr(), blk, blk, t_out.data_ptr(), stride, st.cuda_stream)
            d.wait(st.cuda_stream)   # the call only enqueues; order the read-back after the results
            out = t_out.cpu().numpy()
        a_o = o.process_u8(x)
        for s in range(S):
            assert bits_equal(out[s, :k], a_o)


def test_full_size_batch_4096_streams(rfm, port, synth):
    """BASELINE config 3 at full width: 4096 streams x 2.4 MS/s.  Size-independent properties: a stream's output
    does not depend on its slot or on its neighbours (replicas of 8 distinct contents are identical, wherever
    they sit), and the exemplars equal the oracle."""
    fs, ds, blk = RATES["2.4M"]
    S, K, nblk = 4096, 8, 2
    base = np.stack([synth.make_station_u8(fs, nblk * blk, stream_id=s)[0] for s in range(K)])
    perm = np.random.default_rng(9).integers(0, K, S)
    perm[:K] = np.arange(K)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=S, max_block_len=blk)
    oracles = [port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds) for _ in range(K)]
    for b in range(nblk):
        x = base[:, b * blk:(b + 1) * blk]
        a = d.process_u8(x[perm])
        ex = [oracles[k].process_u8(x[k]) for k in range(K)]
        for k in range(K):
            rows = a[perm == k]
            assert bits_equal(rows[0], ex[k])
            assert np.all(rows.view(np.uint32) == rows[0].view(np.uint32)[None, :])
    bits = {k: oracles[k].take_bits() for k in range(K)}
    for s in (0, 1, 17, 2047, 4095):
        assert np.array_equal(d.take_bits(s), bits[perm[s]])


def test_device_math_probes(rfm):
    """What the GPU computes for the scalar building blocks (rfm_math.cuh), element by element against libm:
    sin/cos == float(sin/cos(double)) [== x87 fsincos -> float], atan2f == glibc atan2f, phase wraps == the
    reference's double expressions, and the branch-free variants == the exact ones wherever they do not flag."""
    import ctypes as C
    libm = C.CDLL("libm.so.6")
    libm.atan2f.restype = C.c_float
    libm.atan2f.argtypes = [C.c_float, C.c_float]
    rng = np.random.default_rng(21)
    n = 2_000_000
    ph = np.concatenate([(rng.random(n) * 7.0 - 0.2), rng.standard_normal(n // 4) * 40.0]).astype(np.float32)
    want = np.stack([np.sin(ph.astype(np.float64)).astype(np.float32), np.cos(ph.astype(np.float64)).astype(np.float32)], 1)
    for op in (0, 2):
        assert bits_equal(rfm.math_probe(op, ph), want), op
    core = np.abs(ph) < 16
    assert bits_equal(rfm.math_probe(1, ph[core]), want[core])
    # atan2f: scalar form, generic form and branch-free form against glibc
    m = 300_000
    y = np.concatenate([rng.standard_normal(m), rng.standard_normal(m) * 1e-3, rng.standard_normal(m)]).astype(np.float32)
    x = np.concatenate([rng.standard_normal(m), rng.standard_normal(m), rng.standard_normal(m) * 1e-4]).astype(np.float32)
    ref = np.array([libm.atan2f(a, b) for a, b in zip(y.tolist(), x.tolist())], dtype=np.float32)
    assert bits_equal(rfm.math_probe(3, y, x)[:, 0], ref)
    assert bits_equal(rfm.math_probe(5, y, x)[:, 0], ref)
    fast = rfm.math_probe(4, y, x)
    ok = fast[:, 1] == 0
    assert ok.mean() > 0.999 and bits_equal(fast[ok, 0], ref[ok])
    sp = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, 1e-45, 3e38, np.nan, 1e-39, 5e19, 2e-20], dtype=np.float32)
    yy, xx = [np.ascontiguousarray(v.ravel()) for v in np.meshgrid(sp, sp)]
    ref = np.array([libm.atan2f(a, b) for a, b in zip(yy.tolist(), xx.tolist())], dtype=np.float32)
    got = rfm.math_probe(3, yy, xx)[:, 0]
    assert np.all((got.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(got) & np.isnan(ref)))
    fast = rfm.math_probe(4, yy, xx)
    okf = fast[:, 1] == 0
    assert np.array_equal(fast[okf, 0].view(np.uint32), ref[okf].view(np.uint32))
    # branch-free division == __fdiv_rn inside the exponent window (1e9 pairs on the device + structured operands)
    bad, tested = rfm.div_selftest(1_000_000_000)
    assert tested > 300_000_000 and bad == 0, (bad, tested)
    a = (rng.standard_normal(n) * 10.0 ** rng.integers(-20, 20, n)).astype(np.float32)
    b = (rng.standard_normal(n) * 10.0 ** rng.integers(-20, 20, n)).astype(np.float32)
    a[:1000] = 0.0
    a[1000:2000] = -0.0
    b[::7] = 1.0
    q = rfm.math_probe(6, a, b)
    okd = q[:, 1] == 0
    assert okd.mean() > 0.5 and bits_equal(q[okd, 0], rfm.math_probe(7, a, b)[okd, 0])
    assert bits_equal(q[okd, 0], (a[okd].astype(np.float64) / b[okd].astype(np.float64)).astype(np.float32))
    # phase wraps
    p = (rng.random(n) * 20.0 - 7.0).astype(np.float32)
    pd = p.astype(np.float64)
    two_pi = 2.0 * 3.14159265358979323846
    dem = np.where(pd >= two_pi, np.fmod(pd, two_pi), pd).astype(np.float32)
    dem = np.where(dem < 0, (dem.astype(np.float64) + two_pi).astype(np.float32), dem)
    pil = np.where(pd > two_pi, pd - two_pi, pd).astype(np.float32)
    dom = (p >= -6.0) & (p < 12.5)
    ex = rfm.math_probe(10, p)
    assert bits_equal(ex[dom, 0], dem[dom]) and bits_equal(ex[dom & (p > 0), 1], pil[dom & (p > 0)])
    f8, f9 = rfm.math_probe(8, p), rfm.math_probe(9, p)
    assert np.array_equal(f8[:, 1] == 0, dom) and bits_equal(f8[dom, 0], dem[dom])
    d9 = (p < 12.5) & (p > 0)
    assert bits_equal(f9[d9, 0], pil[d9])


def test_device_osc_gain_every_float(rfm):
    """math probe 13: the float-only NCO_OSC gain against the double expression, on the device, for every float of
    [0.45, 1.75] (covers the fast-path domain and both fall-back edges)."""
    lo, hi = np.float32(0.45).view(np.uint32), np.float32(1.75).view(np.uint32)
    q = np.arange(lo, hi + 1, dtype=np.uint32).view(np.float32)
    out = rfm.math_probe(13, q)
    assert bits_equal(out[:, 0], out[:, 1])
    ref = (np.float64(1.95) - q.astype(np.float64)).astype(np.float32)
    assert bits_equal(out[:, 1], ref)


def test_speculation_misses_and_degenerate_inputs_stay_exact(rfm, port, synth):
    """The time-parallel FM-demodulator PLL speculates on a contracting loop (DESIGN.md 3.1).  On pure noise the
    speculation misses routinely and chunks are repaired; on constant input operands hit exact zeros (the sticky-flag
    replay path of the lane kernels).  Either way the result must stay bit-identical to the sequential reference."""
    fs, ds, blk = RATES["2.4M"]
    nblk = 3
    rng = np.random.default_rng(77)
    noise = np.clip(np.rint(127.5 + 40 * rng.standard_normal((nblk * blk, 2))), 0, 255).astype(np.uint8)
    weak = np.clip(np.rint(127.5 + 2.0 * rng.standard_normal((nblk * blk, 2))), 0, 255).astype(np.uint8)
    const = np.full((nblk * blk, 2), 128, dtype=np.uint8)
    alt = const.copy()
    alt[::2, 0] = 127
    good = station("2.4M", nblk)[0]
    iqs = np.stack([noise, weak, const, alt, good])
    S = iqs.shape[0]
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=S, max_block_len=blk)
    oracles = [port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds) for _ in range(S)]
    for b in range(nblk):
        a = d.process_u8(iqs[:, b * blk:(b + 1) * blk])
        for s in range(S):
            r = oracles[s].process_u8(iqs[s, b * blk:(b + 1) * blk])
            assert bits_equal(a[s], r), (b, s)
            assert bits_equal(d.tap("baseband", s), oracles[s].tap("baseband")), (b, s)
            so, sd = oracles[s].status(), d.status(s)
            assert all(np.float32(so[k]).view(np.uint32) == np.float32(sd[k]).view(np.uint32) or
                       (np.isnan(so[k]) and np.isnan(sd[k])) for k in so), (b, s, so, sd)
    for s in range(S):
        assert np.array_equal(oracles[s].take_bits(), d.take_bits(s))
    assert d.demod_repairs() > 0, "pure noise is expected to defeat the speculation now and then"


def test_async_submit_matches_synchronous_call(rfm, port):
    """rfm_decoder_submit_u8 (enqueue only, pinned host buffers) over several blocks == the synchronous entry point."""
    import ctypes as C
    import torch
    fs, ds, blk = RATES["1.2M"]
    S, nblk = 6, 4
    iq, _ = station("1.2M", nblk)
    o = port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    ref = [o.process_u8(iq[b * blk:(b + 1) * blk]) for b in range(nblk)]
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=S, max_block_len=blk, n_groups=3)
    stride = d.max_audio_floats(blk)
    h_in = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(iq.reshape(nblk, 1, blk, 2), (nblk, S, blk, 2)))).pin_memory()
    h_out = torch.zeros((nblk, S, stride), dtype=torch.float32).pin_memory()
    k = C.c_uint32(0)
    ks = []
    for b in range(nblk):
        rc = rfm.lib().rfm_decoder_submit_u8(d._h, C.cast(h_in[b].data_ptr(), C.POINTER(C.c_uint8)), blk,
                                             C.cast(h_out[b].data_ptr(), C.POINTER(C.c_float)), stride, C.byref(k))
        assert rc == 0, rfm.lib().rfm_last_error()
        ks.append(k.value)
    d.synchronize()
    out = h_out.numpy()
    for b in range(nblk):
        for s in range(S):
            assert bits_equal(out[b, s, :ks[b]], ref[b]), (b, s)
    assert np.array_equal(d.take_groups(S - 1), o.take_groups())


@pytest.mark.parametrize("fs,ds,blk,kw", [
    (2.048e6, 9, 65520, {}),                               # decimation the tiled front end is not specialised for
    (1.0e6, 4, 65536, {"usver": True}),                    # 75 us deemphasis (USver)
    (1.0e6, 4, 65536, {"bw_pcm": 12000.0}),                # narrower audio bandwidth: other Lanczos / Kaiser tables
    (1.2e6, 5, 65520, {"tuning_offset": 0.0}),             # no fine-tuner shift
    (1.2e6, 5, 65520, {"tuning_offset": 93750.0}),         # positive shift (table walks the other way)
    (960000.0, 4, 65536, {}),
])
def test_other_configurations(rfm, port, synth, fs, ds, blk, kw):
    """Constructor arguments beyond the BASELINE configs (generic front-end kernel, USver, bandwidth, tuning)."""
    kw = dict(kw)
    off = kw.pop("tuning_offset", -0.15 * fs)
    nblk = 3
    iq, _ = synth.make_station_u8(fs, nblk * blk, stream_id=2, f_off=off)
    o = port.OracleFmDecoder(fs, off, downsample=ds, **kw)
    d = rfm.FmDecoderBatch(fs, off, downsample=ds, n_streams=3, max_block_len=blk, n_groups=2, **kw)
    assert np.array_equal(o.constants()[:51], d.constants()[:51])
    for b in range(nblk):
        x = iq[b * blk:(b + 1) * blk]
        a_o = o.process_u8(x)
        a_d = d.process_u8(np.broadcast_to(x, (3,) + x.shape))
        for s in range(3):
            assert bits_equal(a_d[s], a_o), (b, s)
        for t in ("demod_in", "baseband", "rds_dec", "rds_lp", "rds_mf"):
            assert bits_equal(d.tap(t, 2), oracle_tap(o, t)), (t, b)
    assert np.array_equal(o.take_bits(), d.take_bits(1))
