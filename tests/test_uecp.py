"""SURVEY.md section 8f row N1: RDS groups -> UECP frames (cRDSGroupDecoder, RDSGroupDecoder.cpp) and the transport
framing of cRadioReceiver::AddUECPDataFrame (RadioReceiver.cpp:387-414).  Host integer code: no GPU needed, byte-exact.

Three implementations are compared on the same group streams:
  * the UNMODIFIED reference compiled in place (oracle/ref_uecp.py) -- only where oracle/_ref/ holds it,
  * the Python restatement (oracle/uecp_port.py),
  * the product (librfm: rfm_rdsgroup_*, through the C ABI),
all against tests/golden/uecp_kat.npz (generated from the compiled reference by tests/golden/make_golden_uecp.py).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402
from oracle import ref_uecp, uecp_port  # noqa: E402

rfm = load_package()
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "uecp_kat.npz"))


def unpack(buf: np.ndarray) -> list[bytes]:
    raw, out, i = buf.tobytes(), [], 0
    while i < len(raw):
        n = raw[i] | (raw[i + 1] << 8)
        out.append(raw[i + 2:i + 2 + n])
        i += 2 + n
    return out


def names(buf: np.ndarray) -> list[bytes]:
    raw = buf.tobytes()
    return [raw[i:i + 8] for i in range(0, len(raw), 8)]


def product_frames(groups, setting=None, accept=True):
    frames, nm = [], []
    kw = {"on_frame": frames.append, "on_name": lambda s: (nm.append(s.ljust(8, b"\0")[:8]), accept and not (setting and setting()))[1]}
    if setting is not None:
        kw["setting_active"] = setting
    d = rfm.RdsGroupDecoder(**kw)
    d.decode(groups)
    return d, frames, nm


@pytest.mark.parametrize("case", ["scripted", "fuzz"])
def test_port_matches_golden(case):
    o = uecp_port.OracleGroupDecoder()
    assert o.decode(GOLD[f"{case}_groups"]) == unpack(GOLD[f"{case}_frames"])
    assert o.names == names(GOLD[f"{case}_names"])


@pytest.mark.parametrize("case", ["scripted", "fuzz"])
def test_product_matches_golden(case):
    _, frames, nm = product_frames(GOLD[f"{case}_groups"])
    want = unpack(GOLD[f"{case}_frames"])
    assert len(frames) == len(want)
    for i, (a, b) in enumerate(zip(frames, want)):
        assert a == b, f"frame {i}: {a.hex()} != {b.hex()}"
    assert nm == names(GOLD[f"{case}_names"])


def test_scripted_stream_covers_every_message_element():
    """the fixture exercises each MEC the decoder can emit"""
    mecs = {f[4] for f in unpack(GOLD["scripted_frames"])}
    assert mecs == {0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x0A, 0x0D, 0x1A, 0x30, 0x3A, 0x40, 0x46}


def test_frame_layout_and_crc():
    """ADD ADD SQC MFL message CRC (RDSGroupDecoder.cpp:945-993): SQC counts frames, MFL = message length,
    CRC-16/GENIBUS over everything before it (known answer: '123456789' -> 0xD64E)."""
    assert uecp_port.crc16(b"123456789") == 0xD64E
    for i, f in enumerate(unpack(GOLD["scripted_frames"])):
        assert f[0] == 0 and f[1] == 0 and f[2] == i & 0xFF
        assert f[3] == len(f) - 6
        crc = uecp_port.crc16(f[:-2])
        assert f[-2:] == bytes([crc >> 8, crc & 0xFF])


def test_dialog_open_suppresses_frames():
    """IsSettingActive(): frames are not sent (and SQC does not advance), names still go to SetChannelName"""
    s = GOLD["scripted_groups"]
    n = s.shape[0]
    state = {"on": False}
    frames, nm = [], []
    d = rfm.RdsGroupDecoder(on_frame=frames.append, setting_active=lambda: state["on"],
                            on_name=lambda x: (nm.append(x.ljust(8, b"\0")[:8]), not state["on"])[1])
    o = uecp_port.OracleGroupDecoder()
    fo = []
    for lo, hi, on in ((0, n // 3, False), (n // 3, 2 * n // 3, True), (2 * n // 3, n, False)):
        state["on"] = on
        o.setting_active = on
        d.decode(s[lo:hi])
        fo += o.decode(s[lo:hi])
    want = unpack(GOLD["dialog_frames"])
    assert frames == want and fo == want
    assert nm == names(GOLD["dialog_names"]) and o.names == nm
    assert len(want) < len(unpack(GOLD["scripted_frames"]))


def test_transport_framing():
    """RadioReceiver.cpp:387-414: 0xFE, bytes >= 0xFD escaped as (0xFD, (b & 3) - 1), 0xFF"""
    assert uecp_port.stuff_frame(bytes([0x00, 0xFC, 0xFD, 0xFE, 0xFF, 0x10])) == bytes(
        [0xFE, 0x00, 0xFC, 0xFD, 0x00, 0xFD, 0x01, 0xFD, 0x02, 0x10, 0xFF])
    rng = np.random.default_rng(5)
    for n in (0, 1, 7, 262):
        f = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert rfm.uecp_stuff_frame(f) == uecp_port.stuff_frame(f)
    assert rfm.uecp_stuff_frame(b"") == b"\xfe\xff"


def test_internal_buffer_is_the_framed_stream():
    """without callbacks: the PID-2 byte stream (every frame framed, in order), the accepted PS name kept"""
    s = GOLD["scripted_groups"]
    d = rfm.RdsGroupDecoder()
    d.decode(s)
    want = b"".join(uecp_port.stuff_frame(f) for f in unpack(GOLD["scripted_frames"]))
    got = d.take_uecp(100) + d.take_uecp()
    assert got == want and d.take_uecp() == b""
    assert d.channel_name() == names(GOLD["scripted_names"])[-1]
    # frames are dropped while more than 16384 bytes are pending (RadioReceiver.cpp:389-390)
    d2 = rfm.RdsGroupDecoder()
    d2.decode(GOLD["fuzz_groups"])
    got2 = d2.take_uecp(1 << 20)
    framed = [uecp_port.stuff_frame(f) for f in unpack(GOLD["fuzz_frames"])]
    acc = b""
    for f in framed:
        if len(acc) > 16384:
            break
        acc += f
    assert got2 == acc and len(acc) < sum(map(len, framed))


def test_reset_and_rejected_names():
    s = GOLD["scripted_groups"]
    # SetChannelName returning false: no PS frame, the name is offered again on the next complete cycle
    _, fa, na = product_frames(s[:12], accept=False)
    o = uecp_port.OracleGroupDecoder(accept_name=False)
    assert fa == o.decode(s[:12]) and na == o.names and len(na) >= 2
    assert all(f[4] != 0x02 for f in fa)
    # Reset() keeps the sequence counter and the PTY (RDSGroupDecoder.cpp:140-164 touches neither)
    frames = []
    d = rfm.RdsGroupDecoder(on_frame=frames.append)
    d.decode(s[:8])
    k = len(frames)
    d.reset()
    d.decode(s[:8])
    assert frames[k][2] == k and frames[k][4] == 0x01       # PI again (m_ProgramIdentCode was cleared) ...
    assert all(f[4] != 0x07 for f in frames[k:])            # ... but no second PTY frame


@pytest.mark.skipif(not ref_uecp.available(), reason="compiled reference group decoder not present (oracle/_ref)")
def test_against_compiled_reference_random_streams():
    """fresh random streams (not the committed ones) through the reference itself, the port and the product"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden_uecp as mg
    for seed in (1, 2, 3):
        rng = np.random.default_rng(seed)
        g = np.concatenate([mg.fuzz(rng, 3000), mg.scripted(rng), mg.fuzz(rng, 3000)])
        r = ref_uecp.RefGroupDecoder()
        want = r.decode(g)
        wn = r.take_names()
        o = uecp_port.OracleGroupDecoder()
        assert o.decode(g) == want and o.names == wn
        _, frames, nm = product_frames(g)
        assert frames == want and nm == wn


def test_random_streams_match_golden():
    """the streams of test_against_compiled_reference_random_streams through the port and the product, against the
    frames and names stored for them in tests/golden/ref_cases.npz (checked against the original where it is built)"""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden_uecp as mg
    import make_golden_ref_cases as mr
    want = np.load(os.path.join(ROOT, "tests", "golden", "ref_cases.npz"))["uecp_sha"]
    for k, seed in enumerate((1, 2, 3)):
        rng = np.random.default_rng(seed)
        g = np.concatenate([mg.fuzz(rng, 3000), mg.scripted(rng), mg.fuzz(rng, 3000)])
        o = uecp_port.OracleGroupDecoder()
        assert mr.frames_sha(o.decode(g), o.names) == want[k]
        _, frames, nm = product_frames(g)
        assert mr.frames_sha(frames, nm) == want[k]


@pytest.mark.skipif(not ref_uecp.available(), reason="compiled reference group decoder not present (oracle/_ref)")
def test_golden_is_what_the_reference_produces():
    for case in ("scripted", "fuzz"):
        r = ref_uecp.RefGroupDecoder()
        assert r.decode(GOLD[f"{case}_groups"]) == unpack(GOLD[f"{case}_frames"])
        assert r.take_names() == names(GOLD[f"{case}_names"])


def test_cpp_host_class_drop_in(tmp_path):
    """host/RDSGroupDecoder.h: same constructor / DecodeRDS / Reset as the reference's class, driving a receiver
    object through AddUECPDataFrame / SetChannelName / IsSettingActive (no GPU involved)."""
    import subprocess
    lib_dir = os.path.join(ROOT, "pvr.rtl.radiofm_b200")
    exe = str(tmp_path / "host_rdsgroup_driver")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(lib_dir, "host"),
                           os.path.join(ROOT, "tests", "cpp", "host_rdsgroup_driver.cpp"), "-o", exe,
                           "-L", lib_dir, "-lradiofm_b200", f"-Wl,-rpath,{lib_dir}"])
    GOLD["fuzz_groups"].astype("<u2").tofile(tmp_path / "g.bin")
    out = subprocess.run([exe, str(tmp_path / "g.bin"), str(tmp_path / "f.bin"), str(tmp_path / "n.bin")],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert np.fromfile(tmp_path / "f.bin", dtype=np.uint8).tobytes() == GOLD["fuzz_frames"].tobytes()
    assert np.fromfile(tmp_path / "n.bin", dtype=np.uint8).tobytes() == GOLD["fuzz_names"].tobytes()
