"""Generate tests/golden/ref_cases.npz: the expected values of the tests that compare with the compiled original
(oracle/_ref/), so that the same cases are also checked where the original is not built.

    python tests/golden/make_golden_ref_cases.py

The values come from the original (oracle/ref.py, ref_uecp.py, ref_addon.py) where oracle/_ref/ holds it, and
otherwise from the restatement (oracle/port.py, uecp_port.py, demux_port.py), which the tests pin bit for bit to the
original on these very cases; `source` records which.  tests/test_oracle_port.py::
test_ref_cases_golden_is_what_the_reference_produces regenerates the file from the original wherever it is built and
requires it to be identical.  Arrays longer than a few hundred values are stored as SHA-256 digests.

  stage_<rate>_*   test_port_matches_reference_every_stage: per block the digests of the audio and of every stage
                   tap, the status and stereo flag; the RDS groups and bits at the end
  reset_*          test_port_reset_matches_reference: audio digests of 2 blocks, Reset, 2 blocks; the groups
  noisy_sha        test_port_noisy_and_mono_match_reference: 3 stations x 3 blocks of audio
  rdsdc<j>_*       test_rdsdc_port_vs_ref_every_stage_kind: output rate, per call the output count and digest
  uecp_sha         test_uecp.py::test_against_compiled_reference_random_streams: frames and names per seed
  ref12_*          test_gpu_parity.py::test_against_unmodified_reference: 11 blocks at 1.2 MS/s
  odd_*            test_gpu_parity.py::test_default_rtlsdr_block_at_1200k_and_odd_short_blocks: the 20 block sizes
  demux_*          test_ref_addon.py::test_reference_addon_packets_equal_the_restatement and the add-on leg of
                   test_gpu_demux.py: every DemuxRead packet of 8 blocks, the audio level
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, HERE)
import conftest  # noqa: E402
from oracle import demux_port, port, ref, ref_addon, ref_uecp, uecp_port  # noqa: E402

PATH = os.path.join(HERE, "ref_cases.npz")
STAGE_BLOCKS = {"1.0M": 10, "1.2M": 4, "2.4M": 4, "390k": 6}
NOISY = ({"snr_db": 25.0, "stream_id": 3}, {"mono_tone": (1000.0, 0.5)}, {"stereo": False, "rds": False})
RDSDC = ((4.0e6, 4800.0, False, 100000.0, 16384), (2.4e6, 100000.0, False, -57000.0, 8192),
         (50.0e6, 100000.0, True, -7.0e6, 32000), (50.0e6, 100000.0, True, 0.0, 12800))
ODD_SIZES = [65536] * 9 + [100, 333, 1000, 47, 4096, 65521, 777, 20000, 41, 65535, 4097]
DEMUX_BLOCKS = 8


def sha(a) -> str:
    """float32 arrays bit for bit (the tests' bits_equal), bytes as they are"""
    b = bytes(a) if isinstance(a, (bytes, bytearray)) else np.ascontiguousarray(a, dtype=np.float32).tobytes()
    return hashlib.sha256(b).hexdigest()


def packets_sha(packets) -> str:
    """DemuxRead packets: id, pts, duration, then the audio bits (id 1) or the UECP bytes (id 2)"""
    h = hashlib.sha256()
    for sid, pts, dur, data in packets:
        h.update(np.array([sid], np.int32).tobytes() + np.array([pts, dur], np.float64).tobytes())
        if sid == 1:
            h.update(np.ascontiguousarray(data, dtype=np.float32).tobytes())
        elif sid == 2:
            h.update(bytes(data))
    return h.hexdigest()


def frames_sha(frames, names) -> str:
    h = hashlib.sha256()
    for f in frames:
        h.update(len(f).to_bytes(4, "little") + bytes(f))
    h.update(b"|" + b"".join(bytes(n) for n in names))
    return h.hexdigest()


def _decoder(use_ref, fs, ds):
    return (ref.RefFmDecoder if use_ref else port.OracleFmDecoder)(fs, -0.15 * fs, downsample=ds)


def _block(use_ref, d, x8):
    """audio and stage taps of one ProcessStream call"""
    if use_ref:
        return d.process_staged(ref.u8_to_cf32(x8))
    a = d.process_u8(x8)
    return a, d.taps()


def make(use_ref: bool) -> dict:
    out = {"source": np.array("reference" if use_ref else "restatement")}
    for rate, nblk in STAGE_BLOCKS.items():
        fs, ds, blk = conftest.RATES[rate]
        iq, _ = conftest.station(rate, nblk)
        d = _decoder(use_ref, fs, ds)
        digests, status, stereo = [], [], []
        for b in range(nblk):
            a, t = _block(use_ref, d, iq[b * blk:(b + 1) * blk])
            digests.append([sha(a)] + [sha(t[name]) for name in ref.TAP_NAMES])
            status.append([float(v) for v in d.status().values()])
            stereo.append(bool(t["stereo"]))
        out[f"stage_{rate}_sha"] = np.array(digests)
        out[f"stage_{rate}_status"] = np.array(status, dtype=np.float32)
        out[f"stage_{rate}_stereo"] = np.array(stereo)
        out[f"stage_{rate}_groups"] = d.take_groups()
        out[f"stage_{rate}_bits"] = d.take_bits()

    fs, ds, blk = conftest.RATES["1.0M"]
    iq, _ = conftest.station("1.0M", 4)
    d = _decoder(use_ref, fs, ds)
    digests = []
    for b in range(4):
        if b == 2:
            d.reset()
        digests.append(sha(d.process_u8(iq[b * blk:(b + 1) * blk])))
    out["reset_sha"], out["reset_groups"] = np.array(digests), d.take_groups()

    synth = __import__("radiofm_b200.synth", fromlist=["x"])
    noisy = []
    for kw in NOISY:
        iq, _ = synth.make_station_u8(fs, 3 * blk, **kw)
        d = _decoder(use_ref, fs, ds)
        noisy.append([sha(d.process_u8(iq[b * blk:(b + 1) * blk])) for b in range(3)])
    out["noisy_sha"] = np.array(noisy)

    L = ref.lib() if use_ref else port.lib()
    pre = "ref_" if use_ref else "rfo_"
    for j, (in_rate, max_bw, wfm, freq, n) in enumerate(RDSDC):
        rng = np.random.default_rng(11)
        h = getattr(L, pre + "rdsdc_create")()
        getattr(L, pre + "rdsdc_set_frequency")(h, np.float32(freq))
        r = getattr(L, pre + ("rdsdc_set_wfm_data_rate" if wfm else "rdsdc_set_data_rate"))(h, np.float32(in_rate),
                                                                                            np.float32(max_bw))
        ks, digests = [], []
        for _ in range(3):
            x = (rng.standard_normal((n, 2)) * 0.3).astype(np.float32)
            y = np.zeros_like(x)
            k = getattr(L, pre + "rdsdc_process")(h, n, x.ctypes.data_as(port._f32p), y.ctypes.data_as(port._f32p))
            ks.append(k)
            digests.append(sha(y[:k]))
        getattr(L, pre + "rdsdc_destroy")(h)
        out[f"rdsdc{j}_rate"], out[f"rdsdc{j}_k"], out[f"rdsdc{j}_sha"] = np.float32(r), np.array(ks), np.array(digests)

    import make_golden_uecp as mg
    digests = []
    for seed in (1, 2, 3):
        rng = np.random.default_rng(seed)
        g = np.concatenate([mg.fuzz(rng, 3000), mg.scripted(rng), mg.fuzz(rng, 3000)])
        if use_ref:
            r = ref_uecp.RefGroupDecoder()
            frames = r.decode(g)
            names = r.take_names()
        else:
            o = uecp_port.OracleGroupDecoder()
            frames = o.decode(g)
            names = o.names
        digests.append(frames_sha(frames, names))
    out["uecp_sha"] = np.array(digests)

    fs, ds, blk = conftest.RATES["1.2M"]
    iq, _ = conftest.station("1.2M", 11)
    d = _decoder(use_ref, fs, ds)
    out["ref12_sha"] = np.array([sha(d.process_u8(iq[b * blk:(b + 1) * blk])) for b in range(11)])
    out["ref12_bits"], out["ref12_groups"] = d.take_bits(), d.take_groups()

    iq, _ = conftest.station("1.2M", 12)
    d = _decoder(use_ref, fs, ds)
    digests, pos = [], 0
    for n in ODD_SIZES:
        digests.append(sha(d.process_u8(iq[pos:pos + n])))
        pos += n
    out["odd_sha"], out["odd_bits"], out["odd_groups"] = np.array(digests), d.take_bits(), d.take_groups()

    fs, ds, blk = conftest.RATES["1.0M"]
    iq, _ = conftest.station("1.0M", DEMUX_BLOCKS)
    if use_ref:
        a = ref_addon.RefAddon(100.0e6)
        assert a.open()
        for b in range(DEMUX_BLOCKS):
            a.feed(iq[b * blk:(b + 1) * blk], short_read_after_next=(b == 1))
        packets, level = a.read_all(), a.audio_level()
        a.close()
        a.destroy()
    else:
        om = demux_port.OracleDemux(fs, -0.15 * fs, downsample=ds)
        for b in range(DEMUX_BLOCKS):
            om.write_u8(iq[b * blk:(b + 1) * blk])
        packets = []
        while (p := om.read()) is not None:
            packets.append(p)
        level = om.audio_level
    out["demux_sha"], out["demux_audio_level"] = np.array(packets_sha(packets)), np.float32(level)
    out["demux_ids"] = np.array([p[0] for p in packets], dtype=np.int32)
    return out


def reference_available() -> bool:
    return ref.available() and ref_uecp.available() and ref_addon.available()


if __name__ == "__main__":
    np.savez_compressed(PATH, **make(reference_available()))
    print("wrote", PATH, os.path.getsize(PATH), "bytes")
