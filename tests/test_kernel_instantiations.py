"""Every compiled kernel instantiation against the oracle, and an audit that each one is really launched.

1. The inventory (CPU): every __global__ symbol of the sm_100a objects (cuobjdump + cu++filt, as
   test_cubin_resources.py reads them) must have a row in INSTANTIATIONS, and every row must name a symbol of the
   build.  A row names the case of this file that launches the instantiation and compares its output with the CPU
   oracle, or the reason it cannot be reached through the C ABI.  A new template axis without a case fails here,
   before any GPU time is spent.
2. The cases (GPU): each reaches its instantiations through public arguments only -- format (dtype), shared capture,
   IQ correction, NCO, fir_fused, sample rates and downsample, row pitch and base offset of device input, block
   length, stream and row counts -- and compares with the oracle: port.OracleFmDecoder, the oracle's CRDSDownConvert
   and cFreqShift, oracle/scan.py, oracle/iqcorr.py and the port's filters.  The format conversion, the IQ correction
   and the NCO are exact float32 operations restated in numpy (to_cf32, iqcorr.apply, nco.Nco) and feed the oracle.
3. The audit (GPU): the cases run under torch.profiler with CUDA activities; every kernel name it records must map to
   a symbol of the inventory, and every instantiation a row marks as tested must have been launched by its case.
"""
from __future__ import annotations

import functools
import glob
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import bits_equal
from oracle import iqcorr, nco as onco
from test_iq_formats import to_cf32, welch_psd_iq

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "pvr.rtl.radiofm_b200", "csrc", "build")
CUDA_BIN = "/usr/local/cuda/bin"
CUOBJDUMP = shutil.which("cuobjdump") or os.path.join(CUDA_BIN, "cuobjdump")
CUFILT = shutil.which("cu++filt") or os.path.join(CUDA_BIN, "cu++filt")

# the cases (test functions of this file) the table refers to
EXACT = "test_decoder_exact"
FUSED = "test_decoder_fused"
LANES = "test_decoder_lanes_partition"
DC = "test_downconvert_chain"
FS = "test_freqshift_mix"
SCAN = "test_scan_spectrum"
EST = "test_iq_estimate"
PRIM = "test_filter_primitives"
CASES = (EXACT, FUSED, LANES, DC, FS, SCAN, EST, PRIM)

R_PROBE = ("reason: the device-math probe behind rfm_math_probe, a test hook with no chain output to compare; "
           "launched and checked against the host restatement by test_gpu_parity.py::test_device_math_probes")
R_DIV = ("reason: the division self-test behind rfm_div_selftest, a test hook that checks itself on the device "
         "(test_host_math.py); it has no oracle output to compare")

# normalised symbol -> the case that launches it and compares it with the oracle, or "reason: ..."
#   EXACT: bit for bit against port.OracleFmDecoder.  Front ends: k_front_tma / k_front_cs8_tma for u8 / s8 rows a
#   tensor map can describe (ds 1, 5, 11; 16-byte base and pitch, n % 4 == 0), k_front_tiled for every other row of
#   ds 1, 4, 5, 11, k_front for the other downsample factors.  Resampler tiles: GB follows the baseband rate over the
#   PCM rate (8: 125 and 390.625 kHz, 6: 218 kHz, 4: 250 kHz, 3: 300 kHz, 2: 333 kHz, 1: 500 kHz at 8 kHz PCM).
#   k_rotfir<1>: the 15 kHz audio LP has 5 taps at 8 kHz PCM.  k_rds_front: RDS blocks whose length is not a multiple
#   of 8 (and the 390.625 kHz chain); k_rds_front3 otherwise.
#   FUSED: fir_fused = 1, inside the north-star tolerances, RDS bits identical, and not bit-identical.
#   LANES: the immediate-barrier lanes kernel, launched when the decoder runs in an SM partition (lanes_sms).
INSTANTIATIONS = {
    # rfm_downconvert.o
    "k_dc_osc": DC,
    "k_dc_osc_fill": DC,
    "k_dc_chain<0,0,0,0>": DC,
    "k_dc_chain<0,0,0,1>": DC,
    "k_dc_chain<0,0,1,0>": DC,
    "k_dc_chain<0,0,1,1>": DC,
    "k_dc_chain<0,1,0,0>": DC,
    "k_dc_chain<0,1,0,1>": DC,
    "k_dc_chain<0,1,1,0>": DC,
    "k_dc_chain<0,1,1,1>": DC,
    "k_dc_chain<1,0,0,0>": DC,
    "k_dc_chain<1,0,0,1>": DC,
    "k_dc_chain<1,0,1,0>": DC,
    "k_dc_chain<1,0,1,1>": DC,
    "k_dc_chain<1,1,0,0>": DC,
    "k_dc_chain<1,1,0,1>": DC,
    "k_dc_chain<1,1,1,0>": DC,
    "k_dc_chain<1,1,1,1>": DC,
    "k_dc_chain<2,0,0,0>": DC,
    "k_dc_chain<2,0,0,1>": DC,
    "k_dc_chain<2,0,1,0>": DC,
    "k_dc_chain<2,0,1,1>": DC,
    "k_dc_chain<2,1,0,0>": DC,
    "k_dc_chain<2,1,0,1>": DC,
    "k_dc_chain<2,1,1,0>": DC,
    "k_dc_chain<2,1,1,1>": DC,
    "k_dc_chain<3,0,0,0>": DC,
    "k_dc_chain<3,0,0,1>": DC,
    "k_dc_chain<3,0,1,0>": DC,
    "k_dc_chain<3,0,1,1>": DC,
    "k_dc_chain_uniform<0,0,51,0,0>": DC,
    "k_dc_chain_uniform<0,0,51,0,1>": DC,
    "k_dc_chain_uniform<0,0,51,1,0>": DC,
    "k_dc_chain_uniform<0,0,51,1,1>": DC,
    "k_dc_chain_uniform<0,1,51,0,0>": DC,
    "k_dc_chain_uniform<0,1,51,0,1>": DC,
    "k_dc_chain_uniform<0,1,51,1,0>": DC,
    "k_dc_chain_uniform<0,1,51,1,1>": DC,
    "k_dc_chain_uniform<1,0,51,0,0>": DC,
    "k_dc_chain_uniform<1,0,51,0,1>": DC,
    "k_dc_chain_uniform<1,0,51,1,0>": DC,
    "k_dc_chain_uniform<1,0,51,1,1>": DC,
    "k_dc_chain_uniform<1,1,51,0,0>": DC,
    "k_dc_chain_uniform<1,1,51,0,1>": DC,
    "k_dc_chain_uniform<1,1,51,1,0>": DC,
    "k_dc_chain_uniform<1,1,51,1,1>": DC,
    "k_dc_chain_uniform<2,0,51,0,0>": DC,
    "k_dc_chain_uniform<2,0,51,0,1>": DC,
    "k_dc_chain_uniform<2,0,51,1,0>": DC,
    "k_dc_chain_uniform<2,0,51,1,1>": DC,
    "k_dc_chain_uniform<2,1,51,0,0>": DC,
    "k_dc_chain_uniform<2,1,51,0,1>": DC,
    "k_dc_chain_uniform<2,1,51,1,0>": DC,
    "k_dc_chain_uniform<2,1,51,1,1>": DC,
    "k_dc_chain_uniform<3,0,51,0,0>": DC,
    "k_dc_chain_uniform<3,0,51,0,1>": DC,
    "k_dc_chain_uniform<3,0,51,1,0>": DC,
    "k_dc_chain_uniform<3,0,51,1,1>": DC,
    # rfm_freqshift.o
    "k_fs_phase": FS,
    "k_fs_mix<0,0,0>": FS,
    "k_fs_mix<0,0,1>": FS,
    "k_fs_mix<0,1,0>": FS,
    "k_fs_mix<0,1,1>": FS,
    "k_fs_mix<1,0,0>": FS,
    "k_fs_mix<1,0,1>": FS,
    "k_fs_mix<1,1,0>": FS,
    "k_fs_mix<1,1,1>": FS,
    "k_fs_mix<2,0,0>": FS,
    "k_fs_mix<2,0,1>": FS,
    "k_fs_mix<2,1,0>": FS,
    "k_fs_mix<2,1,1>": FS,
    "k_fs_mix<3,0,0>": FS,
    "k_fs_mix<3,0,1>": FS,
    # rfm_iqcorr.o
    "k_iq_stats<0>": EST,
    "k_iq_stats<1>": EST,
    "k_iq_stats<2>": EST,
    "k_iq_stats<3>": EST,
    "k_iq_stats_reduce<double>": EST,
    "k_iq_stats_reduce<longlong>": EST,
    # rfm_kernels.o
    "k_audio_tail": EXACT,
    "k_demod_fix": EXACT,
    "k_demod_repair": EXACT,
    "k_demod_spec": EXACT,
    "k_osc": EXACT,
    "k_rds_front": EXACT,
    "k_rds_pll": EXACT,
    "k_rds_slice": EXACT,
    "k_res_taps": EXACT,
    "k_resample": PRIM,
    "k_tails": EXACT,
    "k_bb_lanes<0,0,0,0>": EXACT,
    "k_bb_lanes<0,1,0,0>": LANES,
    "k_front<0>": EXACT,
    "k_front<1>": EXACT,
    "k_front<2>": EXACT,
    "k_front<3>": EXACT,
    "k_front_cs8_tma<1,0>": EXACT,
    "k_front_cs8_tma<1,1>": FUSED,
    "k_front_cs8_tma<11,0>": EXACT,
    "k_front_cs8_tma<11,1>": FUSED,
    "k_front_cs8_tma<5,0>": EXACT,
    "k_front_cs8_tma<5,1>": FUSED,
    "k_front_tail<0>": EXACT,
    "k_front_tail<1>": EXACT,
    "k_front_tail<2>": EXACT,
    "k_front_tail<3>": EXACT,
    "k_front_tiled<0,1,2>": EXACT,
    "k_front_tiled<0,1,3>": EXACT,
    "k_front_tiled<0,11,2>": EXACT,
    "k_front_tiled<0,11,3>": EXACT,
    "k_front_tiled<0,4,2>": EXACT,
    "k_front_tiled<0,4,3>": EXACT,
    "k_front_tiled<0,5,2>": EXACT,
    "k_front_tiled<0,5,3>": EXACT,
    "k_front_tiled<1,1,0>": EXACT,
    "k_front_tiled<1,1,1>": EXACT,
    "k_front_tiled<1,11,0>": EXACT,
    "k_front_tiled<1,11,1>": EXACT,
    "k_front_tiled<1,4,0>": EXACT,
    "k_front_tiled<1,4,1>": EXACT,
    "k_front_tiled<1,5,0>": EXACT,
    "k_front_tiled<1,5,1>": EXACT,
    "k_front_tma<1,0>": EXACT,
    "k_front_tma<1,1>": FUSED,
    "k_front_tma<11,0>": EXACT,
    "k_front_tma<11,1>": FUSED,
    "k_front_tma<5,0>": EXACT,
    "k_front_tma<5,1>": FUSED,
    "k_if_level<0>": EXACT,
    "k_if_level<1>": EXACT,
    "k_if_level<2>": EXACT,
    "k_if_level<3>": EXACT,
    "k_rds_front3<15,19,35>": EXACT,
    "k_rds_front3<15,23,43>": EXACT,
    "k_resample_tiled<1,0>": EXACT,
    "k_resample_tiled<1,1>": FUSED,
    "k_resample_tiled<2,0>": EXACT,
    "k_resample_tiled<2,1>": FUSED,
    "k_resample_tiled<3,0>": EXACT,
    "k_resample_tiled<3,1>": FUSED,
    "k_resample_tiled<4,0>": EXACT,
    "k_resample_tiled<4,1>": FUSED,
    "k_resample_tiled<6,0>": EXACT,
    "k_resample_tiled<6,1>": FUSED,
    "k_resample_tiled<8,0>": EXACT,
    "k_resample_tiled<8,1>": FUSED,
    "k_rotfir<0>": PRIM,
    "k_rotfir<1>": EXACT,
    "k_rotfir<2>": PRIM,
    "k_rotfir_lanes<0,0>": EXACT,
    "k_rotfir_lanes<0,1>": FUSED,
    "k_rotfir_lanes<1,0>": EXACT,
    "k_rotfir_lanes<1,1>": FUSED,
    "k_rotfir_lanes<2,0>": EXACT,
    "k_rotfir_lanes<2,1>": FUSED,
    # rfm_primitives.o
    "k_downsample_real_int": PRIM,
    "k_join_v": PRIM,
    "k_split": PRIM,
    "k_to_v": PRIM,
    "k_iir<0>": PRIM,
    "k_iir<1>": PRIM,
    "k_iir<2>": PRIM,
    # rfm_probe.o
    "k_div_selftest": R_DIV,
    "k_probe": R_PROBE,
    # rfm_scan.o
    "k_scan_reduce": SCAN,
    "k_scan_psd<0,0>": SCAN,
    "k_scan_psd<0,1>": SCAN,
    "k_scan_psd<1,0>": SCAN,
    "k_scan_psd<1,1>": SCAN,
    "k_scan_psd<2,0>": SCAN,
    "k_scan_psd<2,1>": SCAN,
    "k_scan_psd<3,0>": SCAN,
    "k_scan_psd<3,1>": SCAN,

}


# ---------------------------------------------------------------------------------------------------------------------
# 1. inventory and names
# ---------------------------------------------------------------------------------------------------------------------
def _template_args(s: str) -> list[str]:
    """'<(int)0, (bool)1>' -> ['0', '1']: casts, bool words, integer suffixes and whitespace normalised."""
    out, depth, cur = [], 0, ""
    for ch in s[1:-1]:
        depth += ch in "<("
        depth -= ch in ">)"
        if ch == "," and depth == 0:
            out.append(cur)
            cur = ""
        else:
            cur += ch
    out.append(cur)
    norm = []
    for a in out:
        a = re.sub(r"^\s*\((?:int|bool|unsigned int|unsigned|long|char)\)", "", a.strip())
        a = {"true": "1", "false": "0"}.get(a, a)
        a = re.sub(r"^(-?\d+)[uUlL]*$", r"\1", a)
        norm.append(re.sub(r"\s+", "", a))
    return norm


def normalise(name: str) -> str | None:
    """A demangled kernel name (cu++filt's or the profiler's spelling) -> 'k_name<a,b>' ; None if it names no k_ kernel
    of this project."""
    m = re.search(r"(?:^|[\s:*&(])(k_\w+)", name)
    if not m:
        return None
    ident, rest = m.group(1), name[m.end():]
    if not rest.startswith("<"):
        return ident
    depth = 0
    for i, ch in enumerate(rest):
        depth += ch == "<"
        depth -= ch == ">"
        if depth == 0:
            return ident + "<" + ",".join(_template_args(rest[:i + 1])) + ">"
    return None


def _demangle(names: list[str]) -> list[str]:
    r = subprocess.run([CUFILT], input="\n".join(names) + "\n", capture_output=True, text=True, check=True)
    out = r.stdout.split("\n")[:len(names)]
    assert len(out) == len(names)
    return out


@functools.lru_cache(maxsize=1)
def inventory() -> dict[str, str]:
    """normalised symbol -> demangled name, for every __global__ function of the compiled objects."""
    objs = sorted(glob.glob(os.path.join(BUILD, "*.o")))
    if not objs or not os.path.exists(CUOBJDUMP) or not os.path.exists(CUFILT):
        pytest.skip("no compiled objects / cuobjdump / cu++filt (run __graft_entry__.build())")
    inv = {}
    for o in objs:
        r = subprocess.run([CUOBJDUMP, "--dump-resource-usage", o], capture_output=True, text=True)
        if r.returncode != 0:
            continue  # host-only object
        mangled = re.findall(r"^\s*Function\s+(\S+):", r.stdout, flags=re.M)
        if not mangled:
            continue
        for d in _demangle(mangled):
            key = normalise(d)
            assert key, f"{os.path.basename(o)}: kernel {d!r} is not named k_*"
            assert key not in inv, f"two instantiations normalise to {key}: {inv[key]!r} and {d!r}"
            inv[key] = d
    return inv


def test_every_instantiation_has_exactly_one_row():
    inv = inventory()
    missing = sorted(set(inv) - set(INSTANTIATIONS))
    extra = sorted(set(INSTANTIATIONS) - set(inv))
    assert not missing, "instantiations without a row (add a case that launches them, or the reason they cannot be " \
                        f"reached): {missing}"
    assert not extra, f"rows naming no symbol of the build: {extra}"
    for k, v in INSTANTIATIONS.items():
        assert v in CASES or (v.startswith("reason: ") and len(v) > 40), (k, v)


def test_profiler_spellings_normalise_to_the_inventory_names():
    """The profiler demangles with the C++ runtime: '(anonymous namespace)', 'false' / 'true', plain integers."""
    inv = inventory()
    cupti = {
        "void (anonymous namespace)::k_dc_chain_uniform<0, true, 51, false, true>((anonymous namespace)::DcParams, "
        "rfm::DcTapsPk<51>, rfm::IqCorr, (anonymous namespace)::DcNco)": "k_dc_chain_uniform<0,1,51,0,1>",
        "void rfm::k_front_cs8_tma<11, true>(rfm::FrontParams, rfm::FrontCoef, CUtensorMap_st, unsigned int, "
        "unsigned int)": "k_front_cs8_tma<11,1>",
        "void (anonymous namespace)::k_iq_stats_reduce<long long>(long long const*, unsigned int, long long*)":
            "k_iq_stats_reduce<longlong>",
        "rfm::k_demod_spec(rfm::DemodSpecParams)": "k_demod_spec",
        "(anonymous namespace)::k_scan_reduce(float const*, unsigned int, double, float*)": "k_scan_reduce",
        "void rfm::k_resample_tiled<6u, false>(rfm::ResampleParams, unsigned int)": "k_resample_tiled<6,0>",
    }
    for name, want in cupti.items():
        assert normalise(name) == want and want in inv, (name, normalise(name))
    assert normalise("void at::native::vectorized_elementwise_kernel<4, at::native::FillFunctor<float>>(int)") is None
    for d in inventory().values():
        assert normalise(d) in INSTANTIATIONS


# ---------------------------------------------------------------------------------------------------------------------
# 2. launch recording
# ---------------------------------------------------------------------------------------------------------------------
LAUNCHED: dict[str, set] = {}     # case -> normalised symbols its runs launched
FOREIGN: dict[str, set] = {}      # case -> profiler kernel names that map to no symbol


def _torch():
    import torch
    return torch


def _kernel_names(prof) -> list[str]:
    torch = _torch()
    cuda = torch.autograd.DeviceType.CUDA
    names = []
    for e in prof.profiler.kineto_results.events():
        if e.device_type() == cuda:
            names.append(e.name())
    return names


def _record(case: str, names: list[str]):
    inv = inventory()
    mangled = [n for n in names if n.startswith("_Z")]
    if mangled:
        dm = dict(zip(mangled, _demangle(mangled)))
        names = [dm.get(n, n) for n in names]
    for n in names:
        if n.startswith(("Memcpy", "Memset")):
            continue
        key = normalise(n)
        if key in inv:
            LAUNCHED.setdefault(case, set()).add(key)
        else:
            FOREIGN.setdefault(case, set()).add(n)


@pytest.fixture
def launches(request):
    """Runs the case under torch.profiler (CUDA activities) and records the kernels it launched under its name."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    case = request.node.originalname
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        yield
        torch.cuda.synchronize()
    _record(case, _kernel_names(prof))


# ---------------------------------------------------------------------------------------------------------------------
# 3. the cases
# ---------------------------------------------------------------------------------------------------------------------
_ESZ = {"u8": 2, "s8": 2, "s16": 4, "cf32": 8}
_DT = {"u8": np.uint8, "s8": np.int8, "s16": np.int16, "cf32": np.float32}


def _as_format(u8: np.ndarray, fmt: str, seed: int = 0) -> np.ndarray:
    """u8 IQ -> the same signal in fmt's container (s8: exact shift; s16 / cf32: with low-order dither)."""
    rng = np.random.default_rng(seed)
    v = u8.astype(np.int32) - 128
    if fmt == "u8":
        return u8
    if fmt == "s8":
        return v.astype(np.int8)
    if fmt == "s16":
        # clipped: -128 * 256 + dither can fall below -32768, and a cast would wrap it to the other rail
        return np.clip(v * 256 + rng.integers(-128, 128, size=v.shape), -32768, 32767).astype(np.int16)
    return (to_cf32(u8) + rng.standard_normal(u8.shape).astype(np.float32) * np.float32(1e-3)).astype(np.float32)


def _device_rows(torch, rows: np.ndarray, pitch: int, off: int):
    """[R, n, 2] host rows -> (tensor, pointer of row 0): rows `pitch` samples apart, `off` samples past the base."""
    R, n = rows.shape[:2]
    flat = np.zeros((R * pitch + off + 8, 2), dtype=rows.dtype)
    for r in range(R):
        flat[off + r * pitch:off + r * pitch + n] = rows[r]
    t = torch.from_numpy(flat).cuda()
    return t, t.data_ptr() + off * rows.dtype.itemsize * 2


def _layout(i: int, n: int, fmt: str) -> tuple[int, int] | None:
    """Entry point of call i: None = host arrays; else (row pitch, base offset) of device rows: a 16-byte pitch
    multiple at an aligned base, or an odd pitch one sample past it."""
    if i % 3 == 0:
        return None
    if i % 3 == 1:
        q = 16 // _ESZ[fmt] if _ESZ[fmt] < 16 else 1
        return ((n + 1 + q - 1) // q) * q, 0
    return n + 3 if (n + 3) % 2 else n + 4, 1


# ---- decoder -------------------------------------------------------------------------------------------------------
# label -> (fs_if, downsample, fs_pcm, bw_pcm, streams)
DECODERS = {
    "1.0M/4": (1.0e6, 4, 48000.0, 15000.0, 33),
    "2.4M/11": (2.4e6, 11, 48000.0, 15000.0, 31),
    "1.2M/5": (1.2e6, 5, 48000.0, 15000.0, 1),
    "390k/1": (390625.0, 1, 48000.0, 15000.0, 65),
    "1.0M/3": (1.0e6, 3, 48000.0, 15000.0, 2),
    "1.0M/8": (1.0e6, 8, 48000.0, 15000.0, 1),
    "1.2M/4": (1.2e6, 4, 48000.0, 15000.0, 3),
    "1.0M/2@8k": (1.0e6, 2, 8000.0, 3000.0, 1),
}


def _lengths(ds: int) -> list[int]:
    """A TMA-friendly block, the minimum (the input FIR order), one output short of / at / past a 384-output front-end
    tile, and a long block (several demodulator chunks)."""
    t = 384 * ds
    return [4 * t, 8 * ds, t - ds, t, t + ds, 24000]


def _rds_stage_lengths(rfm, label: str) -> list[int]:
    """Lengths of the planned RDS decimate-by-2 stages (rfm_plan_constants: ..., audio LP taps, stage count, six
    lengths); 11 is the fixed 11-tap stage, 3 the CIC3."""
    fs, ds, pcm, bw = DECODERS[label][:4]
    s = rfm.plan_constants(fs, -0.15 * fs, pcm, bw, ds)
    return [int(v) for v in s[45:45 + int(s[44])]]


def _rds_skipped_blocks(stages: list[int], ds: int, lens: list[int]) -> list[int]:
    """The blocks whose RDS branch the decoder skips (PlanBlock, rfm_api.cu; DESIGN.md section 7): a fixed 11-tap or
    CIC3 stage fed an odd count or fewer than 18 samples reads outside its input in the reference, where the result is
    undefined, so the library leaves RDS untouched for that block and the oracle's bits are not comparable after it."""
    pos, skipped = 0, []
    for i, n in enumerate(lens):
        nb = (n - pos + ds - 1) // ds if pos < n else 0
        pos = pos + nb * ds - n
        m = nb
        for L in stages:
            if L in (3, 11):
                if m % 2 or m < 18:
                    skipped.append(i)
                    break
                m //= 2
            else:
                m = m // 2 if m < L else (m + 1) // 2
    return skipped


def _rds_lengths(stages: list[int], ds: int) -> list[int]:
    """Blocks of about 4, 2 and 6 front-end tiles, each lengthened until no stage of the RDS chain skips it."""
    lens = []
    for n in (4 * 384 * ds, 2 * 384 * ds + 1, 24000):
        while _rds_skipped_blocks(stages, ds, lens + [n]):
            n += 1
        lens.append(n)
    return lens


@functools.lru_cache(maxsize=None)
def _station(fs: float, n: int) -> np.ndarray:
    from conftest import load_package
    load_package()
    import importlib
    synth = importlib.import_module("radiofm_b200.synth")
    return synth.make_station_u8(fs, n)[0]


def _decoder_rows(label: str, fmt: str, S: int, lens: list[int]) -> np.ndarray:
    fs = DECODERS[label][0]
    total = sum(lens)
    base = _station(fs, total + 1013 * S)
    u8 = np.stack([base[1013 * s:1013 * s + total] for s in range(S)])
    return _as_format(u8, fmt, seed=S)


def _run_decoder(rfm, port, label, fmt, S, fused=0, lanes_sms=0, lens=None):
    """Feeds the decoder and S oracles call by call; yields (block, audio [S] rows, oracle rows), then (None, None,
    decoder status, oracle status) per stream.  The RDS bits are compared at the end unless a block skipped the RDS
    branch (_rds_skipped_blocks)."""
    torch = _torch()
    fs, ds, pcm, bw = DECODERS[label][:4]
    lens = lens or _lengths(ds)
    compare_bits = not _rds_skipped_blocks(_rds_stage_lengths(rfm, label), ds, lens)
    raw = _decoder_rows(label, fmt, S, lens)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, pcm, bw, downsample=ds, n_streams=S, max_block_len=max(lens), device=0,
                           lanes_sms=lanes_sms, fir_fused=fused)
    oracles = [port.OracleFmDecoder(fs, -0.15 * fs, pcm, bw, downsample=ds) for _ in range(S)]
    pos = 0
    for i, n in enumerate(lens):
        x = np.ascontiguousarray(raw[:, pos:pos + n])
        pos += n
        lay = _layout(i, n, fmt)
        if lay is None:
            got = d.process_iq(x)
        else:
            t, ptr = _device_rows(torch, x, *lay)
            stride = (d.max_audio_floats(n) + 1) & ~1
            a = torch.empty((S, stride), dtype=torch.float32, device="cuda")
            k = d.process_iq_device(fmt, ptr, lay[0], n, a.data_ptr(), stride)
            d.synchronize()
            got = a.cpu().numpy()[:, :k]
            del t
        want = [o.process_u8(x[s]) if fmt == "u8" else o.process_cf32(to_cf32(x[s])) for s, o in enumerate(oracles)]
        yield i, n, got, want
    for s, o in enumerate(oracles):
        if compare_bits:
            bits = o.take_bits()
            assert bits.size > 0 and np.array_equal(d.take_bits(s), bits), (label, fmt, s, "RDS bits")
        yield None, None, d.status(s), o.status()
    d.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["u8", "s8", "s16", "cf32"])
@pytest.mark.parametrize("label", list(DECODERS))
def test_decoder_exact(rfm, port, launches, label, fmt):
    """Audio, status and RDS bits bit for bit over the edge-shaped blocks of _lengths; where those make the RDS chain's
    fixed 11-tap / CIC3 stage skip a block, a second run with blocks it accepts compares the RDS bits."""
    fs, ds = DECODERS[label][:2]
    S = DECODERS[label][4]
    stages = _rds_stage_lengths(rfm, label)
    runs = [_lengths(ds)]
    if _rds_skipped_blocks(stages, ds, runs[0]):
        runs.append(_rds_lengths(stages, ds))
        assert not _rds_skipped_blocks(stages, ds, runs[1])
    for lens in runs:
        for i, n, got, want in _run_decoder(rfm, port, label, fmt, S, lens=lens):
            if i is None:
                assert all(np.float32(want[k]) == np.float32(got[k]) for k in want), (label, fmt, got, want)
                continue
            for s in range(S):
                assert bits_equal(got[s], want[s]), (label, fmt, lens, "block", i, n, "stream", s)


@pytest.mark.gpu
@pytest.mark.parametrize("label,fmt", [("2.4M/11", "u8"), ("2.4M/11", "s8"), ("1.2M/5", "u8"), ("1.2M/5", "s8"),
                                       ("390k/1", "u8"), ("390k/1", "s8"), ("1.0M/4", "s16"), ("1.0M/3", "u8"),
                                       ("1.0M/8", "u8"), ("1.2M/4", "cf32"), ("1.0M/2@8k", "u8")])
def test_decoder_fused(rfm, port, launches, label, fmt):
    """fir_fused = 1: audio within 1e-4 of full scale, L+R within 1e-5, L-R within 2e-4, the same stereo decisions and
    RDS bits -- and not bit-identical, so a switch that does nothing fails."""
    exact = True
    worst = 0.0
    ds = DECODERS[label][1]
    stages = _rds_stage_lengths(rfm, label)
    lens = _lengths(ds)
    if _rds_skipped_blocks(stages, ds, lens):
        lens = _rds_lengths(stages, ds)
    for i, n, got, want in _run_decoder(rfm, port, label, fmt, 2, fused=1, lens=lens):
        if i is None:
            assert got["stereo"] == want["stereo"], (label, fmt)
            continue
        for s in range(2):
            assert got[s].shape == want[s].shape, (label, fmt, i, s)
            if want[s].size == 0:
                continue
            exact &= bits_equal(got[s], want[s])
            worst = max(worst, float(np.max(np.abs(got[s] - want[s]))))
            g, r = got[s].reshape(-1, 2).astype(np.float64), want[s].reshape(-1, 2).astype(np.float64)
            assert float(np.max(np.abs((g[:, 0] + g[:, 1]) - (r[:, 0] + r[:, 1])))) <= 1e-5, (label, fmt, i, s)
            assert float(np.max(np.abs((g[:, 0] - g[:, 1]) - (r[:, 0] - r[:, 1])))) <= 2e-4, (label, fmt, i, s)
    assert 0.0 < worst <= 1e-4 and not exact, (label, fmt, worst)


@pytest.mark.gpu
def test_decoder_lanes_partition(rfm, port, launches):
    """An SM partition for the lanes (rfm_config::lanes_sms) selects the immediate-barrier lanes kernel."""
    for i, n, got, want in _run_decoder(rfm, port, "1.0M/4", "u8", 33, lanes_sms=16):
        if i is None:
            assert all(np.float32(want[k]) == np.float32(got[k]) for k in want)
            continue
        for s in range(33):
            assert bits_equal(got[s], want[s]), ("block", i, n, "stream", s)


# ---- wideband down-converter ---------------------------------------------------------------------------------------
class OracleDc:
    """The oracle's CRDSDownConvert (DownConvert.cpp:271-727) of one row."""

    def __init__(self, port, freq, in_rate, max_bw, wfm):
        import ctypes as C
        self.C, self.L = C, port.lib()
        self.h = self.L.rfo_rdsdc_create()
        self.L.rfo_rdsdc_set_frequency(self.h, np.float32(freq))
        fn = self.L.rfo_rdsdc_set_wfm_data_rate if wfm else self.L.rfo_rdsdc_set_data_rate
        fn(self.h, np.float32(in_rate), np.float32(max_bw))

    def process(self, x):
        P = lambda a: a.ctypes.data_as(self.C.POINTER(self.C.c_float))   # noqa: E731
        z = np.array(x, dtype=np.float32, order="C").reshape(-1, 2)
        y = np.zeros((z.shape[0], 2), dtype=np.float32)
        k = self.L.rfo_rdsdc_process(self.h, z.shape[0], P(z), P(y))
        return y[:k].copy()

    def __del__(self):
        self.L.rfo_rdsdc_destroy(self.h)


def _capture(fmt: str, shape, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if fmt == "u8":
        return rng.integers(0, 256, size=shape, dtype=np.uint8)
    if fmt == "s8":
        return rng.integers(-128, 128, size=shape).astype(np.int8)
    if fmt == "s16":
        return rng.integers(-20000, 20000, size=shape).astype(np.int16)
    return (rng.standard_normal(shape) * 0.3).astype(np.float32)


CORR = (np.float32(0.01), np.float32(-0.02), np.float32(1.05), np.float32(0.03))
# plan -> (in_rate, max_bw, wfm, lengths): the uniform HB51 chain (5120-sample tiles; 6400 is its minimum; the long
# call is cut into time chunks) and a generic HB15 / HB23 / HB51 chain (2048-sample tiles; 400 is its minimum)
DC_PLANS = {
    "uniform": (50.0e6, 100000.0, True, [10240, 6400, 10240 - 128, 10240 + 128, 24 * 5120]),
    "generic": (2.4e6, 100000.0, False, [2048, 400, 2048 - 8, 2048 + 8, 65536]),
}
DC_CROSSINGS = [(f, sh, c, n) for f in ("u8", "s8", "s16", "cf32") for sh in (False, True) for c in (False, True)
                for n in (False, True) if not (f == "cf32" and sh)]


def _crossing_id(x):
    f, sh, c, n = x
    return f"{f}-{'shared' if sh else 'rows'}{'-corr' if c else ''}{'-nco' if n else ''}"


@pytest.mark.gpu
@pytest.mark.parametrize("crossing", DC_CROSSINGS, ids=[_crossing_id(x) for x in DC_CROSSINGS])
@pytest.mark.parametrize("plan", list(DC_PLANS))
def test_downconvert_chain(rfm, port, launches, plan, crossing):
    torch = _torch()
    fmt, shared, corr, use_nco = crossing
    fs, bw, wfm, lens = DC_PLANS[plan]
    k = DC_CROSSINGS.index(crossing)
    rows = [1, 31, 33, 65][k % 4] if plan == "generic" else [1, 3][k % 2]
    osc = [(-1) ** r * (r + 1) * fs / 97.0 for r in range(rows)]
    nfreq = [fs / 2 - r * fs / max(rows, 2) for r in range(rows)]   # +in_rate / 2 (the edge) down towards -in_rate / 2
    dc = rfm.DownConvertBatch(osc, fs, bw, wfm=wfm, max_len=max(lens), device=0)
    oracles = [OracleDc(port, f, fs, bw, wfm) for f in osc]
    ncos = [onco.Nco(f, np.float32(fs)) for f in nfreq] if use_nco else None
    if corr:
        dc.set_iq_correction(rfm.IqCorrection(*CORR))
    if use_nco:
        dc.set_nco(nfreq)
    for i, n in enumerate(lens):
        raw = _capture(fmt, (n, 2) if shared else (rows, n, 2), seed=1000 * i + k)
        m = n >> dc.n_stages
        lay = _layout(i, n, fmt)
        if lay is None:
            got = dc.process_iq(raw, shared_capture=shared)
        else:
            t, ptr = _device_rows(torch, raw[None] if shared else raw, *lay)
            out = torch.empty((rows, m, 2), dtype=torch.float32, device="cuda")
            assert dc.process_iq_device(fmt, shared, ptr, lay[0], out.data_ptr(), m, n) == m
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            del t
        for r in range(rows):
            x = to_cf32(raw if shared else raw[r])
            if corr:
                x = iqcorr.apply(x, *CORR)
            if use_nco:
                x = ncos[r].mix(x)
            assert bits_equal(got[r], oracles[r].process(x)), (plan, crossing, "call", i, n, "row", r)


# ---- freqshift -----------------------------------------------------------------------------------------------------
FS_CROSSINGS = [(f, sh, c) for f in ("u8", "s8", "s16", "cf32") for sh in (False, True) for c in (False, True)
                if not (f == "cf32" and sh)]


@pytest.mark.gpu
@pytest.mark.parametrize("crossing", FS_CROSSINGS,
                         ids=[f"{f}-{'shared' if sh else 'rows'}{'-corr' if c else ''}" for f, sh, c in FS_CROSSINGS])
def test_freqshift_mix(rfm, port, launches, crossing):
    """cFreqShift rows (FreqShift.h:12-27) against the oracle's, phases carried over calls of 1, 255, 256, 257 and
    40000 samples."""
    import ctypes as C
    torch = _torch()
    fmt, shared, corr = crossing
    k = FS_CROSSINGS.index(crossing)
    rows = [1, 31, 33, 65][k % 4]
    fs = 2.4e6
    freqs = [(r - rows // 2) * 7919.0 for r in range(rows)]
    lens = [256, 1, 255, 257, 40000]
    f = rfm.FreqShiftBatch(freqs, fs, max_len=max(lens), device=0)
    if corr:
        f.set_iq_correction(rfm.IqCorrection(*CORR))
    L = port.lib()
    hs = [L.rfo_freqshift_create(np.float32(q), np.float32(fs)) for q in freqs]
    for i, n in enumerate(lens):
        raw = _capture(fmt, (n, 2) if shared else (rows, n, 2), seed=77 + 1000 * i + k)
        lay = _layout(i, n, fmt)
        if lay is None:
            got = f.process_iq(raw, shared_capture=shared)
        else:
            t, ptr = _device_rows(torch, raw[None] if shared else raw, *lay)
            out = torch.empty((rows, n, 2), dtype=torch.float32, device="cuda")
            f.process_iq_device(fmt, shared, ptr, lay[0], out.data_ptr(), n, n)
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            del t
        for r, h in enumerate(hs):
            x = to_cf32(raw if shared else raw[r])
            if corr:
                x = iqcorr.apply(x, *CORR)
            x = np.array(x, dtype=np.float32, order="C")
            L.rfo_freqshift_process(h, x.ctypes.data_as(C.POINTER(C.c_float)), n)
            assert bits_equal(got[r], x), (crossing, "call", i, n, "row", r)
    for h in hs:
        L.rfo_freqshift_destroy(h)
    f.close()


# ---- scan spectrum -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("corr", [False, True])
@pytest.mark.parametrize("fmt", ["u8", "s8", "s16", "cf32"])
def test_scan_spectrum(rfm, launches, fmt, corr):
    """The averaged spectrum against oracle/scan.py's float64 Welch spectrum of the converted (and corrected) samples,
    within 1e-6 of the total power.  4096-sample segments 2048 apart, 32 segments per CTA: exactly four CTAs, and
    129 segments plus a partial hop (a fifth CTA of one segment); both longer than one demodulator call of the scan's
    confirmation, the shortest capture it accepts."""
    for n in (4096 + 2048 * 127, 4096 + 2048 * 128 + 1000):
        cap = _capture(fmt, (n, 2), seed=n + corr)
        s = rfm.BandScan(2.4e6, -1.0e6, 200000.0, 11, min_snr_db=200.0, device=0,
                         iq_correction=rfm.IqCorrection(*CORR) if corr else None)
        s.run(cap)
        x = to_cf32(cap)
        ref = welch_psd_iq(iqcorr.apply(x, *CORR) if corr else x)
        psd = s.spectrum().astype(np.float64)
        assert psd.shape == ref.shape
        assert float(np.max(np.abs(psd - ref))) <= 1e-6 * float(np.sum(ref)), (fmt, corr, n)
        assert s.stations() == []
        s.close()


# ---- IQ estimate ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["u8", "s8", "s16", "cf32"])
def test_iq_estimate(rfm, launches, fmt):
    """rfm_iq_estimate against oracle/iqcorr.py: the integer formats bit for bit, cf32 within 1e-12 of the float64
    sums before the float rounding; one sample, one short of / at / past one CTA's 16384 samples, several CTAs."""
    torch = _torch()
    for n in (1, 16383, 16384, 16385, 3 * 16384 + 1):
        rng = np.random.default_rng(n)
        cap = _capture(fmt, (n, 2), seed=n)
        if fmt != "cf32":     # a DC offset and an imbalance to estimate
            cap = np.clip(cap.astype(np.int32) * np.array([1, 0.8]) + [5, -3], np.iinfo(cap.dtype).min,
                          np.iinfo(cap.dtype).max).astype(cap.dtype)
        host = rfm.estimate_iq_correction(cap)
        t = torch.from_numpy(np.ascontiguousarray(cap)).cuda()
        torch.cuda.synchronize()
        dev = rfm.estimate_iq_correction(t)
        assert dev == host, (fmt, n)
        if fmt != "cf32":
            want = iqcorr.estimate(cap)
            assert host == rfm.IqCorrection(*want[:4], bool(want[4])), (fmt, n, host, want)
            continue
        ref = iqcorr.coefficients_float64(cap)
        for name, got, r in zip(("dc_i", "dc_q", "a", "b"), (host.dc_i, host.dc_q, host.a, host.b), ref[:4]):
            lo, hi = sorted((float(r) * (1 - 1e-12), float(r) * (1 + 1e-12)))
            assert np.float32(lo) <= got <= np.float32(hi), (n, name, got, r)
        del rng


# ---- filter primitives ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_filter_primitives(rfm, port, launches):
    """rfm_iir (real, complex, two rows), rfm_fir under 8 taps (thread per output) and at 9 (lane per row),
    cDownsampleFilter's complex integer (generic front end), real integer and real fractional (untiled resampler) forms,
    against the port, over calls with carried state; 33 and 65 rows."""
    import ctypes as C
    P = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))   # noqa: E731
    L = port.lib()
    rng = np.random.default_rng(31)
    rows = 33
    iir = rfm.IirFilterBatch(rows, max_len=4096)
    assert iir.init(2, 1187.5, 500.0, 31250.0)
    hs = [L.rfo_iir_create() for _ in range(rows)]
    for h in hs:
        assert L.rfo_iir_init(h, 2, 1187.5, 500.0, 31250.0)
    for n in (1, 31, 32, 33, 4096):
        x = rng.standard_normal((rows, n)).astype(np.float32)
        a, b = rng.standard_normal((2, rows, n)).astype(np.float32)
        z = rng.standard_normal((rows, n, 2)).astype(np.float32)
        y, (ya, yb), yz = iir.process_real(x), iir.process_two(a, b), iir.process_complex(z)
        for r, h in enumerate(hs):
            rx, ra, rb, rz = x[r].copy(), a[r].copy(), b[r].copy(), z[r].copy()
            L.rfo_iir_process_real(h, P(rx), n)
            L.rfo_iir_process_two(h, P(ra), P(rb), n)
            L.rfo_iir_process_complex(h, P(rz), n)
            assert bits_equal(y[r], rx) and bits_equal(ya[r], ra) and bits_equal(yb[r], rb), ("iir", r, n)
            assert bits_equal(yz[r], rz), ("iir complex", r, n)
    for h in hs:
        L.rfo_iir_destroy(h)
    for ntaps, rows in ((5, 65), (7, 1), (9, 33)):
        taps = rng.standard_normal(ntaps).astype(np.float32)
        real, cplx = rfm.FirFilterBatch(rows, max_len=4096), rfm.FirFilterBatch(rows, max_len=4096)
        nt = cplx.init_lp(ntaps, 1.0, 30.0, 5000.0, 12000.0, 48000.0)
        real.init_const(taps, 48000.0)
        hr, hc = [L.rfo_fir_create() for _ in range(rows)], [L.rfo_fir_create() for _ in range(rows)]
        for h, g in zip(hr, hc):
            L.rfo_fir_init_const(h, ntaps, P(taps), 48000.0)
            assert L.rfo_fir_init_lp(g, ntaps, 1.0, 30.0, 5000.0, 12000.0, 48000.0) == nt
        for n in (1, ntaps - 1, ntaps, ntaps + 1, 511, 512, 513, 4096):
            x = rng.standard_normal((rows, n)).astype(np.float32)
            a, b = rng.standard_normal((2, rows, n)).astype(np.float32)
            z = rng.standard_normal((rows, n, 2)).astype(np.float32)
            y, (ya, yb), yz = real.process_real(x), cplx.process_two(a, b), cplx.process_complex(z)
            for r in range(rows):
                rx, ra, rb, rz = x[r].copy(), a[r].copy(), b[r].copy(), z[r].copy()
                L.rfo_fir_process_real(hr[r], P(rx), n)
                L.rfo_fir_process_two(hc[r], P(ra), P(rb), n)
                L.rfo_fir_process_complex(hc[r], P(rz), n)
                assert bits_equal(y[r], rx), ("fir real", ntaps, r, n)
                assert bits_equal(ya[r], ra) and bits_equal(yb[r], rb) and bits_equal(yz[r], rz), ("fir", ntaps, r, n)
        for h in hr + hc:
            L.rfo_fir_destroy(h)
        real.close()
        cplx.close()
    rows = 3
    for order, cutoff, ds, integer, cplx in ((24, 0.2, 3.0, True, True), (40, 0.12, 5.0, True, False),
                                             (500, 15000.0 / 500000.0, 500000.0 / 48000.0, False, False)):
        f = rfm.DownsampleFilterBatch(rows, order, cutoff, ds, integer, max_len=8192)
        hs = [L.rfo_downsample_create(order, cutoff, ds, int(integer)) for _ in range(rows)]
        for n in (order, 4097, 8192, 1001):
            x = rng.standard_normal((rows, n, 2) if cplx else (rows, n)).astype(np.float32)
            y = f.process_complex(x) if cplx else f.process_real(x)
            for r, h in enumerate(hs):
                ref = np.zeros((n, 2) if cplx else n, dtype=np.float32)
                fn = L.rfo_downsample_process_complex if cplx else L.rfo_downsample_process_real
                m = fn(h, P(x[r].copy()), P(ref), n)
                assert y.shape[1] == m and bits_equal(y[r], ref[:m]), ("downsample", order, ds, r, n)
        for h in hs:
            L.rfo_downsample_destroy(h)
        f.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. the audit
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_profiler_sees_the_librarys_launches(rfm, port):
    """CUPTI (through torch.profiler) records the kernels of this ctypes-loaded library, on its own streams and inside
    the decoder's SM partition (green contexts): otherwise the audit below could not see them."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        rfm.estimate_iq_correction(_capture("s16", (5000, 2), seed=1))
        d = rfm.FmDecoderBatch(1.0e6, -0.15e6, downsample=4, n_streams=2, max_block_len=8192, device=0, lanes_sms=16)
        d.process_iq(np.stack([_station(1.0e6, 8192)] * 2))
        d.synchronize()
        d.close()
        torch.cuda.synchronize()
    seen = {normalise(n) for n in _kernel_names(prof)}
    assert "k_iq_stats<2>" in seen and "k_iq_stats_reduce<longlong>" in seen, sorted(map(str, seen))
    assert "k_bb_lanes<0,1,0,0>" in seen and "k_front_tiled<1,4,0>" in seen, sorted(map(str, seen))


@pytest.mark.gpu
def test_launch_audit(capsys):
    """Runs after the cases: every profiler kernel name maps to a symbol of the build, and every instantiation the
    table marks as tested was launched by its case.  Prints the table with the outcome of each row."""
    inv = inventory()
    if not LAUNCHED:
        pytest.skip("no case of this file ran in this session")
    foreign = {c: sorted(v) for c, v in FOREIGN.items() if v}
    assert not foreign, f"profiler kernel names that map to no instantiation: {foreign}"
    missing = sorted(k for k, c in INSTANTIATIONS.items() if c in CASES and k not in LAUNCHED.get(c, ()))
    width = max(map(len, inv))
    with capsys.disabled():
        print(f"\n{len(inv)} instantiations:")
        for k in sorted(inv):
            c = INSTANTIATIONS.get(k, "?")
            state = ("launched by " if k in LAUNCHED.get(c, ()) else "NOT LAUNCHED by ") + c if c in CASES else c
            print(f"  {k:<{width}}  {state}")
    assert not missing, f"instantiations their case never launched: {missing}"
