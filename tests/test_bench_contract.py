"""The JSON lines bench.py printed on the B200 (committed under profiles/) carry every key the driver's contract
names; the metric / unit / workload are BASELINE.json's.  CPU-only: reads the committed lines."""
from __future__ import annotations

import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(name):
    with open(os.path.join(ROOT, "profiles", name)) as f:
        return json.loads(f.read().strip().splitlines()[-1])


def test_b200_arm_line():
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    for name, n in (("r01_bench.json", 1), ("r01_bench_n2.json", 2), ("r01_bench_n8.json", 8)):
        d = load(name)
        assert d["metric"] == base["metric"] and d["unit"] == "MS/s" and d["n_gpus"] == n
        for k in ("value", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                  "config", "roofline", "e2e", "gpu_launches", "clocks"):
            assert k in d, (name, k)
        assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
        assert d["warmup"] >= 3 and d["gpu_launches"] > 0 and d["data"] == "synthetic" and d["dtype"] == "f32"
        assert "workload" in d["config"] and "4096" in d["config"]["workload"] and "l2" in d["config"]
        r = d["roofline"]
        assert r["bound"] in ("hbm", "tensor") and r["unit"] == "GB/s"
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1.2
        e = d["e2e"]
        assert e["unit"] == "MS/s" and e["h2d_bytes_per_step"] == 4096 * 65472 * 2 and e["d2h_bytes_per_step"] > 0
        assert 0 < e["value"] < d["value"]                  # PCIe-bound: below the device-resident figure
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if n == 1:
            c = d["cpu_baseline"]
            assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
            assert r["traffic"] is None or r["traffic"] > 0


def test_reference_arm_line():
    d = load("r01_bench_reference.json")
    b = load("r01_bench.json")
    assert d["impl"] == "reference" and d["metric"] == b["metric"] and d["unit"] == b["unit"]
    assert d["config"]["workload"] == b["config"]["workload"] and d["higher_is_better"] is True
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] == "reference"
    assert d["gpu_launches"] == 0


def test_dump_outputs_fits_the_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the whole batch where it fits, else the same seeded sample of streams on every run,
    within the rank's share of the byte budget, .npy headers included; rows carry their global stream ids."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    rng = np.random.default_rng(0)
    a = rng.standard_normal((64, 1000)).astype(np.float32)
    ga = [rng.integers(0, 65536, (k % 3, 4)).astype(np.uint16) for k in range(64)]
    bench.dump_outputs(str(tmp_path / "a"), a, ga, 0, 0, 1)
    assert sorted(os.listdir(tmp_path / "a")) == ["audio.npy", "rds_group_counts.npy", "rds_groups.npy", "stream_ids.npy"]
    assert np.array_equal(np.load(tmp_path / "a" / "audio.npy"), a)
    assert np.array_equal(np.load(tmp_path / "a" / "rds_groups.npy"), np.concatenate(ga).astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "a" / "rds_group_counts.npy"), [len(g) for g in ga])
    assert np.array_equal(np.load(tmp_path / "a" / "stream_ids.npy"), np.arange(64))
    # the largest audio that fills one rank's share (1 MB / 2) to the byte once the headers are counted
    share = (1 << 20) // 2
    rows = 300
    width = ((share - 4 * bench.NPY_HEADER) // rows - 16) // 4
    b = rng.standard_normal((1024, width)).astype(np.float32)
    gb = [np.zeros((0, 4), np.uint16)] * 1024
    for d in ("b1", "b2"):
        bench.dump_outputs(str(tmp_path / d), b, gb, 1024, 1, 2)
    files = sorted(os.listdir(tmp_path / "b1"))
    assert files == ["audio_rank1.npy", "rds_group_counts_rank1.npy", "rds_groups_rank1.npy", "stream_ids_rank1.npy"]
    assert sum(os.path.getsize(tmp_path / "b1" / f) for f in files) <= share
    ids, got = np.load(tmp_path / "b1" / "stream_ids_rank1.npy"), np.load(tmp_path / "b1" / "audio_rank1.npy")
    assert ids.dtype == np.float64 and got.dtype == np.float32 and ids.size == rows
    assert np.all(np.diff(ids) > 0) and ids.min() >= 1024 and ids.max() < 2048
    assert np.array_equal(got, b[ids.astype(np.int64) - 1024])
    for f in files:
        assert np.array_equal(np.load(tmp_path / "b1" / f), np.load(tmp_path / "b2" / f))


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_block(tmp_path, rfm):
    """bench.py --dump-outputs end to end: the dumped audio is what the decoder returns for the last timed block of the
    seeded batch (after the warm-up and the timed blocks before it), the groups what it decoded by then."""
    import importlib
    import subprocess
    import sys
    import torch
    import bench
    S, K, W = 8, 8, 3
    out = tmp_path / "d"
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(K), "--warmup", str(W), "--streams",
                    str(S), "--no-extras", "--no-cpu", "--no-e2e", "--no-prof", "--dump-outputs", str(out)],
                   check=True, cwd=str(tmp_path), capture_output=True)
    synth_device = importlib.import_module("radiofm_b200.synth_device")
    nres = min(K + W, 12)   # bench.py --resident-blocks default
    iq = synth_device.make_batch_u8(torch, S, bench.FS, nres * bench.BLK, torch.device("cuda", 0)).cpu().numpy()
    d = rfm.FmDecoderBatch(bench.FS, -0.15 * bench.FS, downsample=bench.DS, n_streams=S, max_block_len=bench.BLK, device=0)
    for i in range(W + K):
        b = i % nres
        a = d.process_u8(iq[:, b * bench.BLK:(b + 1) * bench.BLK])
    got = np.load(out / "audio.npy")
    assert got.dtype == np.float32 and got.shape == a.shape and np.array_equal(got.view(np.uint32), a.view(np.uint32))
    groups = [d.take_groups(s) for s in range(S)]
    assert sum(len(g) for g in groups) > 0
    assert np.array_equal(np.load(out / "rds_group_counts.npy"), [len(g) for g in groups])
    assert np.array_equal(np.load(out / "rds_groups.npy"), np.concatenate(groups).astype(np.float64))
    assert np.array_equal(np.load(out / "stream_ids.npy"), np.arange(S))
