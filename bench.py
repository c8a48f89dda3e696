#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native IQ -> audio (+RDS) chain.

    python bench.py --gpus N --steps K --warmup W            (driver contract; torchrun for N > 1)
    python bench.py --impl reference ...                      (the reference's own CPU chain, same workload)
    python bench.py ... --dump-outputs DIR                    (also writes the last timed step's audio and the RDS groups to DIR)

Workload (BASELINE.json configs[3], the one the metric is quoted on; fits one GPU): a batch of 4096 independent
synthetic 2.4 MS/s u8 IQ streams (stereo + RDS stations), full chain.  One step = one 65472-sample block of every
stream (268 M complex samples).  Multi-GPU: streams shard across ranks with no collective (weak scaling:
4096 streams per GPU); torch.distributed is used only for the barrier and the max-over-ranks timing.

value  : complex MS/s with the IQ blocks already resident in HBM (device-pointer C-ABI entry point).
e2e    : the same through the host-buffer C-ABI call (rfm_decoder_process_u8): pinned host IQ in, audio out,
         H2D / D2H inside the timed region, RDS bits drained to the host block-sync at the end.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS, DS, BLK = 2.4e6, 11, 65472          # SURVEY.md section 8: 2.4 MS/s, downsample 11, block 65472
STREAMS_PER_GPU = 4096
BYTES_PER_SAMPLE = 2.0 + 8.0 * 48000.0 / FS   # SURVEY.md 8(d): u8 I,Q in + f32 L,R out = 2.160 B / complex sample
METRIC = "demodulated complex MS/s per GPU (stereo+RDS) at 1/2/4/8 B200; % of HBM roofline"

# ncu-derived constants (dram bytes per launch of each kernel, warp instructions per step) live in
# profiles/ncu_constants.json, written by tools/ncu_constants.py from an `ncu --set full` capture and STAMPED with the
# SHA-256 of the kernel sources it was captured from.  They are printed only when the stamp matches the sources this
# run was built from; otherwise roofline.traffic / roofline.issue are null (a stale constant is not a measurement).
def kernel_sources_sha():
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pvr.rtl.radiofm_b200", "csrc")
    for name in sorted(os.listdir(d)):
        if name.endswith((".cu", ".cuh", ".cpp", ".h", ".inc")):
            h.update(name.encode())
            h.update(open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def load_ncu_constants():
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_constants.json")) as f:
            c = json.load(f)
        if c.get("kernel_sources_sha") != kernel_sources_sha():
            return None, f"stale (captured at sources {c.get('kernel_sources_sha')}, commit {c.get('commit')})"
        return c, f"profiles/ncu_constants.json (commit {c.get('commit')}, {c.get('capture')})"
    except Exception as e:
        return None, f"absent ({type(e).__name__})"


SCHEDULERS = 148 * 4


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0: float, t1: float) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 7] or [r for _, r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        f = lambda v: float(v) if v.replace(".", "", 1).isdigit() else None
        sm = [f(r[0]) for r in rows if f(r[0]) is not None]
        pw = [f(r[2]) for r in rows if f(r[2]) is not None]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": f(rows[0][1]),
                "power_w_max": max(pw) if pw else None, "samples": len(rows), "reasons": reasons}


# --------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own chain (oracle/_ref, compiled from /root/reference by oracle/Makefile) or, where
# that library did not travel, the oracle's plain-C restatement.  One decoder per thread, all host cores.
# --------------------------------------------------------------------------------------------------------------
def cpu_chain():
    from oracle import ref, port
    if ref.available():
        return "reference", lambda: ref.RefFmDecoder(FS, -0.15 * FS, downsample=DS)
    return "port", lambda: port.OracleFmDecoder(FS, -0.15 * FS, downsample=DS)


def cpu_input(n_blocks: int) -> np.ndarray:
    from __graft_entry__ import load_package
    load_package()
    import importlib
    synth = importlib.import_module("radiofm_b200.synth")
    iq, _ = synth.make_station_u8(FS, n_blocks * BLK, stream_id=0)
    return iq.reshape(n_blocks, BLK, 2)


def cpu_step(decoders, iq, pool, blocks_per_thread, b0):
    def work(k):
        d = decoders[k]
        for j in range(blocks_per_thread):
            d.process_u8(iq[(b0 + j) % iq.shape[0]])
    list(pool.map(work, range(len(decoders))))
    return len(decoders) * blocks_per_thread * BLK


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, make = cpu_chain()
    cores = len(os.sched_getaffinity(0))
    iq = cpu_input(8)
    decoders = [make() for _ in range(cores)]
    bpt = 64  # blocks per thread per step: ~0.2 s of CPU work per thread per step (with 8 the 24 ms steps measured the
              # thread pool's hand-over as much as the chain: 344 MS/s against the 440 of the 10 s cpu_baseline leg)
    with cf.ThreadPoolExecutor(cores) as pool:
        for w in range(args.warmup):
            cpu_step(decoders, iq, pool, bpt, w * bpt)
        t0 = time.perf_counter()
        samples = 0
        for k in range(args.steps):
            samples += cpu_step(decoders, iq, pool, bpt, (args.warmup + k) * bpt)
        dt = time.perf_counter() - t0
    v = samples / dt / 1e6
    peak, how = load_peaks()
    sample = f"{cores} threads x 1 stream x {bpt} blocks of {BLK} IQ samples per step (ctypes releases the GIL)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": v, "unit": "MS/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(n_gpus):
    return {"workload": f"C4: {STREAMS_PER_GPU} independent 2.4 MS/s u8 IQ streams per GPU (stereo+RDS stations), "
                        f"one {BLK}-sample block of every stream per step",
            "streams_per_gpu": STREAMS_PER_GPU, "fs_if": FS, "downsample": DS, "block_len": BLK,
            "sharding": f"streams sharded over {n_gpus} GPU(s), no collective",
            "l2": "per-step input (536 MB u8) is larger than L2 (126 MB); a different block every step"}


def cpu_baseline_leg():
    kind, make = cpu_chain()
    cores = len(os.sched_getaffinity(0))
    iq = cpu_input(8)
    decoders = [make() for _ in range(cores)]
    with cf.ThreadPoolExecutor(cores) as pool:
        cpu_step(decoders, iq, pool, 2, 0)
        t0 = time.perf_counter()
        samples, b = 0, 0
        while time.perf_counter() - t0 < 10.0:
            samples += cpu_step(decoders, iq, pool, 64, b)
            b += 64
        dt = time.perf_counter() - t0
    return {"value": samples / dt / 1e6, "unit": "MS/s", "cores": cores, "kind": kind,
            "sample": f"{cores} threads, one decoder each, same 2.4 MS/s stereo+RDS blocks of {BLK} samples, "
                      f"{samples // BLK} blocks in {dt:.1f} s"}


# --------------------------------------------------------------------------------------------------------------
# Extra legs of the same JSON line (VERDICT r01 item 5): the add-on's own call, strong scaling, the wideband config.
# --------------------------------------------------------------------------------------------------------------
def single_stream_leg(rfm, local):
    """The call the add-on actually makes (RadioReceiver.cpp:515-525): ONE stream, 65536 complex samples at 1.0 MS/s,
    blocking cFmDecoder::ProcessStream == rfm_decoder_process_cf32 with host buffers; next to the reference's own
    ProcessStream on one host core (oracle/_ref, cpu_baseline leg)."""
    import importlib
    synth = importlib.import_module("radiofm_b200.synth")
    from oracle import ref, port
    fs, ds, blk, nblk = 1.0e6, 4, 65536, 12
    iq, _ = synth.make_station_u8(fs, nblk * blk, stream_id=0)
    x = port.u8_to_cf32(iq).reshape(nblk, blk, 2)
    d = rfm.FmDecoderBatch(fs, -0.15 * fs, downsample=ds, n_streams=1, max_block_len=blk, device=local)
    ts = []
    for r in range(3):
        for b in range(nblk):
            t0 = time.perf_counter()
            d.process_cf32(x[b][None])
            ts.append((time.perf_counter() - t0) * 1e3)
    d.close()
    gpu_ms = statistics.median(ts[nblk:])
    kind, ref_ms = "port", None
    dec = ref.RefFmDecoder(fs, -0.15 * fs, downsample=ds) if ref.available() else port.OracleFmDecoder(fs, -0.15 * fs, downsample=ds)
    kind = "reference" if ref.available() else "port"
    tr = []
    for r in range(2):
        for b in range(nblk):
            t0 = time.perf_counter()
            dec.process_cf32(x[b])
            tr.append((time.perf_counter() - t0) * 1e3)
    ref_ms = statistics.median(tr[nblk:])
    return {"workload": "1 stream, 65536 complex samples per call at 1.0 MS/s (65.5 ms of signal), host cf32 in, host audio out",
            "api": "rfm_decoder_process_cf32 (blocking; == cFmDecoder::ProcessStream, RadioReceiver.cpp:515-525)",
            "b200_ms_per_call": gpu_ms, "reference_ms_per_call": ref_ms, "reference_kind": kind, "reference_cores": 1,
            "realtime_factor_b200": 65.536 / gpu_ms, "realtime_factor_reference": 65.536 / ref_ms,
            "note": "one stream cannot fill a GPU: every per-stream recurrence runs one lane, so a call costs its dependent "
                    "chain (block latency, ~20 kernel launches); the batch is where the GPU pays"}


def c5_leg(torch, rfm, rank, world, local, barrier, max_over_ranks, steps=12, warmup=3):
    """BASELINE.json configs[4]: one shared 50 MS/s capture, 100 stations on a 200 kHz raster sharded over the ranks
    (no collective; every rank reads the same capture), both mixers.  One step = one demodulator call = 64 front-end
    blocks of 32000 capture samples (41 ms of signal)."""
    import importlib
    synth_device = importlib.import_module("radiofm_b200.synth_device")
    wideband = importlib.import_module("radiofm_b200.wideband")
    shard = importlib.import_module("radiofm_b200.shard")
    FS5, BLK5, BPC5 = 50.0e6, 32000, 64
    n_call, n_st = BLK5 * BPC5, 100
    freqs = [(k - n_st // 2) * 200000.0 for k in range(n_st)]
    lo, hi = shard.shard_range(n_st, rank, world)
    dev = torch.device("cuda", local)
    ncalls = 3
    capture = synth_device.make_wideband_u8(torch, FS5, ncalls * n_call, freqs, dev)
    peak, _ = load_peaks()
    out = {"workload": f"C5: one shared 50 MS/s u8 capture, {n_st} FM stations on a 200 kHz raster sharded by station over "
                       f"{world} GPU(s), mixer + CRDSDownConvert (7 x HB51) + cFmDecoder per station; one step = {BPC5} "
                       f"front-end blocks of {BLK5} samples (41 ms of signal)", "stations": n_st,
           "stations_this_rank": hi - lo, "scaling": "strong"}
    for mixer in ("freqshift", "osc"):
        wb = wideband.WidebandReceiver(torch, freqs[lo:hi], FS5, BLK5, BPC5, mixer=mixer, device=local)
        for i in range(warmup):
            wb.process_device(capture.data_ptr() + 2 * (i % ncalls) * n_call)
        wb.wait()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            nfl = wb.process_device(capture.data_ptr() + 2 * ((warmup + i) % ncalls) * n_call)
        wb.wait()
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / steps
        # front end alone (mixer + decimation chain): CUDA events around one more call of it
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        wb.dc.process_device(1, capture.data_ptr(), n_call, wb.bb.data_ptr(), wb.n_bb, n_call)
        f1.record()
        torch.cuda.synchronize()
        front_ms = f0.elapsed_time(f1)
        algo = 2.0 * n_call + (hi - lo) * nfl * 4.0      # per rank per step: one read of the capture + the audio
        out[mixer] = {"value": n_st * n_call / (ms * 1e-3) / 1e6, "unit": "MS/s (station-samples, whole job)",
                      "ms_per_step": ms, "realtime_factor": (n_call / FS5) / (ms * 1e-3), "front_end_ms": front_ms,
                      "roofline": {"bound": "hbm", "kernel": "k_dc_chain_uniform" + (" + k_dc_osc" if mixer == "osc" else ""),
                                   "achieved": algo / (front_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                   "frac": algo / (front_ms * 1e-3) / 1e9 / peak, "traffic": None,
                                   "note": "FP32-issue-bound (129 un-fused flop per station-sample), the capture is read once "
                                           "from L2 by all stations: DESIGN.md 8.1"}}
        wb.close()
    return out


DUMP_BYTES = 64 << 20
NPY_HEADER = 128   # bytes of an .npy header for arrays of up to two dimensions


def dump_outputs(out_dir, audio, groups, first_stream, rank, world):
    """What the device-resident path delivered by the end of the timed steps, as float32 / float64 .npy files:
      audio.npy             [streams, floats] float32, the audio of the last timed block (interleaved L, R);
      rds_groups.npy        [groups, 4] float64, the RDS groups decoded so far (rfm_decoder_rds_take_groups), the
                            streams' one after another;
      rds_group_counts.npy  [streams] float64, how many of them belong to each stream;
      stream_ids.npy        [streams] float64, the global stream id of each row (first_stream + index in the batch).
    With several GPUs each rank writes <name>_rank<r>.npy.  Where the batch exceeds the rank's share of DUMP_BYTES, a
    fixed seeded sample of its streams is written."""
    sfx = "" if world == 1 else f"_rank{rank}"
    os.makedirs(out_dir, exist_ok=True)
    n = audio.shape[0]
    budget = DUMP_BYTES // world - 4 * NPY_HEADER - sum(g.shape[0] for g in groups) * 4 * 8
    rows = max(0, budget) // (audio[0].nbytes + 16)
    idx = np.arange(n)
    if rows < n:
        idx = np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    picked = [np.asarray(groups[i], dtype=np.float64).reshape(-1, 4) for i in idx]
    out = {"audio": audio[idx], "rds_groups": np.concatenate(picked) if picked else np.zeros((0, 4)),
           "rds_group_counts": np.array([g.shape[0] for g in picked], dtype=np.float64),
           "stream_ids": (first_stream + idx).astype(np.float64)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}{sfx}.npy"), a)


# --------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package
    rfm = load_package()
    import importlib
    synth_device = importlib.import_module("radiofm_b200.synth_device")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    S = args.streams
    K, W = args.steps, args.warmup
    nres = min(K + W, args.resident_blocks)
    iq = synth_device.make_batch_u8(torch, S, FS, nres * BLK, dev, first_stream=rank * S)
    torch.cuda.synchronize()
    dec = rfm.FmDecoderBatch(FS, -0.15 * FS, downsample=DS, n_streams=S, max_block_len=BLK, device=local,
                             n_groups=args.groups, lanes_sms=args.lanes_sms, fir_fused=args.fir_fused)
    stride = dec.max_audio_floats(BLK)
    audio = torch.zeros((S, stride), dtype=torch.float32, device=dev)
    stream = torch.cuda.Stream()
    esz = 2  # bytes per u8 IQ sample

    def step_device(i):
        b = i % nres
        return dec.process_u8_device(iq.data_ptr() + b * BLK * esz, nres * BLK, BLK, audio.data_ptr(), stride,
                                     stream.cuda_stream)

    # ---- value: inputs resident in HBM
    with torch.cuda.stream(stream):
        for i in range(W):
            step_device(i)
        dec.wait(stream.cuda_stream)
    barrier()
    def timed_pass(first_block):
        """K steps, barrier + synchronize on both sides, CUDA events on the caller's stream."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        with torch.cuda.stream(stream):
            e0.record(stream)
            n_out = 0
            th0 = time.perf_counter()
            for i in range(K):
                n_out = step_device(first_block + i)   # only enqueues: consecutive blocks pipeline inside the decoder
            enq = (time.perf_counter() - th0) * 1e3 / K
            dec.wait(stream.cuda_stream)               # the timed region ends when the last block's audio is complete
            e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), n_out, enq

    # pass 1 (the metric): nothing but the K steps between the two events
    launches0 = rfm.launch_count()
    clocks = ClockSampler(local)
    time.sleep(0.25)
    t0 = time.perf_counter()
    ms, nfl, host_enqueue_ms = timed_pass(W)
    t1 = time.perf_counter()
    clk = clocks.stop(t0, t1)
    launches = rfm.launch_count() - launches0
    if args.dump_outputs:
        # pass 2 below rewrites the same audio buffer: take the metric pass's last block now
        dump_outputs(args.dump_outputs, audio[:, :nfl].cpu().numpy(), [dec.take_groups(s) for s in range(S)], rank * S,
                     rank, world)
    # pass 2 (the roofline leg): the same K steps again with every kernel launch bracketed by CUDA events on the
    # stream it is launched on; ~50 extra event records per step cost 3-4 %, which is why it is not the metric pass
    prof, ms_prof = {}, None
    if not args.no_prof:
        dec.set_profiling(True)
        ms_prof, _, _ = timed_pass(W + K)
        prof = dec.profile()
        dec.set_profiling(False)
    repairs = dec.demod_repairs()
    value = world * S * BLK * K / (ms * 1e-3) / 1e6

    # dominant kernel by accumulated device time
    top = max(prof.items(), key=lambda kv: kv[1][0]) if prof else ("none", (0.0, 0))
    top_name, (top_ms, top_n) = top
    peak, how = load_peaks()
    n_groups = max(1, round(top_n / max(K, 1)))
    units_per_launch = S * BLK / n_groups
    avg_ms = top_ms / max(top_n, 1)
    achieved = BYTES_PER_SAMPLE * units_per_launch / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
    ncu_c, ncu_src = load_ncu_constants()
    traffic = None
    if ncu_c and S == STREAMS_PER_GPU and n_groups == 1:
        traffic = ncu_c.get("dram_bytes_per_launch", {}).get(top_name)
    step_traffic = ncu_c.get("dram_bytes_per_step") if (ncu_c and S == STREAMS_PER_GPU) else None
    roofline = {"bound": "hbm", "kernel": top_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": how, "ncu_constants": ncu_src,
                "step_dram_bytes": step_traffic,
                "note": "the chain is latency-bound (one-lane-per-stream pilot PLL recurrence, k_bb_lanes) and FP32-issue-"
                        "bound (bit-exact un-fused FIRs), not HBM-bound: see DESIGN.md sections 3, 3.2",
                "avg_launch_ms": avg_ms, "launches": top_n, "units_per_launch": units_per_launch,
                "algorithmic_bytes_per_unit": BYTES_PER_SAMPLE,
                "chain_achieved": BYTES_PER_SAMPLE * value * 1e6 / 1e9 / world,
                "chain_frac": BYTES_PER_SAMPLE * value * 1e6 / 1e9 / world / peak,
                "timed_pass": "second pass of the same K steps with per-kernel CUDA events (the metric pass carries none)",
                "ms_per_step_with_events": (ms_prof / K) if ms_prof else None,
                "kernel_ms_per_step": {k: round(v[0] / K, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}
    if ncu_c and S == STREAMS_PER_GPU and clk.get("sm_mhz"):
        # the bound that actually binds beside the pilot recurrence: warp-instruction issue slots (SURVEY.md 8d asks for
        # the FP32 figure alongside the HBM one); every FP32 operation of the bit-exact chain is its own instruction
        wi = float(ncu_c["warp_instructions_per_step"])
        issue_peak = SCHEDULERS * float(clk["sm_mhz"]) * 1e6
        roofline["issue"] = {"warp_instructions_per_step": wi, "schedulers": SCHEDULERS,
                             "achieved_per_s": wi / (ms / K * 1e-3), "peak_per_s": issue_peak,
                             "frac": wi / (ms / K * 1e-3) / issue_peak,
                             "source": "ncu smsp__inst_executed.sum over the step's kernels (" + ncu_src + "), one issue "
                                       "slot per scheduler per cycle at the sampled SM clock"}

    # ---- e2e: host buffers through the public host-pointer entry point (its own decoder: stream groups overlap
    # the H2D copy of one group with the kernels / D2H of the others)
    import ctypes as C
    if args.no_e2e:
        if rank == 0:
            print(json.dumps({"value": value, "ms_per_step": ms / K, "host_enqueue_ms_per_step": host_enqueue_ms, "demod_repairs": repairs,
                              "kernel_ms_per_step": roofline["kernel_ms_per_step"]}))
        return
    dec.close()
    dec = rfm.FmDecoderBatch(FS, -0.15 * FS, downsample=DS, n_streams=S, max_block_len=BLK, device=local,
                             n_groups=args.host_groups, lanes_sms=args.lanes_sms)
    nh = min(nres, 2)
    h_iq = torch.empty((nh, S, BLK, 2), dtype=torch.uint8).pin_memory()
    h_iq.copy_(iq.view(S, nres, BLK, 2)[:, :nh].permute(1, 0, 2, 3))
    h_audio = torch.empty((S, stride), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    kout = C.c_uint32(0)
    lib = rfm.lib()

    def step_host(i):
        rc = lib.rfm_decoder_process_u8(dec._h, C.cast(h_iq[i % nh].data_ptr(), C.POINTER(C.c_uint8)), BLK,
                                        C.cast(h_audio.data_ptr(), C.POINTER(C.c_float)), stride, C.byref(kout))
        if rc != 0:
            raise RuntimeError(lib.rfm_last_error().decode())

    for i in range(max(1, W // 2)):
        step_host(i)
    dec.take_groups(0)            # one-time allocations of the drain path (pinned staging) belong to the warm-up
    barrier()
    if os.environ.get("RFM_E2E_PROF"):
        dec.set_profiling(True)
    t0 = time.perf_counter()
    for i in range(K):
        step_host(i)
    groups = dec.take_groups(0)   # drains the RDS bits of every stream to the host block-sync
    if os.environ.get("RFM_E2E_PROF"):
        dec.profile()
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_sync = {"value": world * S * BLK * K / dt / 1e6, "unit": "MS/s", "ms_per_step": dt / K * 1e3,
                "api": "rfm_decoder_process_u8 (blocking: returns with the block's audio on the host) + rfm_decoder_rds_take_groups"}

    # the streaming form of the same public API (rfm_decoder_submit_u8 + rfm_decoder_synchronize): what a producer that
    # has the next block ready uses.  Two pinned host input / output buffers alternate, so the H2D copy of block k+1
    # overlaps the kernels and the D2H of block k.  This is the headline e2e figure; every step still moves its
    # inputs host -> device and its audio device -> host inside the timed region, and the RDS groups of every stream
    # are drained to the host before the clock stops.
    h_audio2 = torch.empty((2, S, stride), dtype=torch.float32).pin_memory()

    def submit_host(i):
        rc = lib.rfm_decoder_submit_u8(dec._h, C.cast(h_iq[i % nh].data_ptr(), C.POINTER(C.c_uint8)), BLK,
                                       C.cast(h_audio2[i % 2].data_ptr(), C.POINTER(C.c_float)), stride, C.byref(kout))
        if rc != 0:
            raise RuntimeError(lib.rfm_last_error().decode())

    for i in range(max(1, W // 2)):
        submit_host(i)
    dec.synchronize()
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        submit_host(i)
    dec.synchronize()
    groups = dec.take_groups(0)
    dt = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e = {"value": world * S * BLK * K / dt / 1e6, "unit": "MS/s", "h2d_bytes_per_step": S * BLK * 2,
           "d2h_bytes_per_step": S * int(kout.value) * 4, "ms_per_step": dt / K * 1e3,
           "api": "rfm_decoder_submit_u8 x K + rfm_decoder_synchronize + rfm_decoder_rds_take_groups (pinned host IQ "
                  "in, host audio out)",
           "blocking": e2e_sync}

    # bare pinned-host -> device copies of the same bytes on every rank at once: the ceiling of any e2e figure on this host
    probe_stream = torch.cuda.Stream()
    d_probe = torch.empty((S, BLK, 2), dtype=torch.uint8, device=dev)
    barrier()
    t0 = time.perf_counter()
    with torch.cuda.stream(probe_stream):
        for i in range(K):
            d_probe.copy_(h_iq[i % nh], non_blocking=True)
    probe_stream.synchronize()
    dt_probe = max_over_ranks(time.perf_counter() - t0)
    barrier()
    del d_probe
    h2d_gbs = world * S * BLK * 2 * K / dt_probe / 1e9
    e2e["h2d_ceiling_gbs"] = h2d_gbs
    e2e["h2d_ceiling_value"] = world * S * BLK * K / dt_probe / 1e6
    e2e["h2d_achieved_gbs"] = e2e["value"] * 1e6 * 2 / 1e9
    e2e["note"] = ("PCIe-bound: h2d_ceiling_* is a bare cudaMemcpyAsync of the same pinned input blocks on all ranks at "
                   "once, nothing else running")
    dec.close()

    # ---- strong scaling (SURVEY.md 8e): 4096 streams in TOTAL over the ranks (the same figure as `value` at N = 1)
    strong = None
    if world > 1:
        Ss = STREAMS_PER_GPU // world
        dec_s = rfm.FmDecoderBatch(FS, -0.15 * FS, downsample=DS, n_streams=Ss, max_block_len=BLK, device=local)
        def step_strong(i):
            return dec_s.process_u8_device(iq.data_ptr() + (i % nres) * BLK * esz, nres * BLK, BLK, audio.data_ptr(), stride,
                                           stream.cuda_stream)
        with torch.cuda.stream(stream):
            for i in range(W):
                step_strong(i)
            dec_s.wait(stream.cuda_stream)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for i in range(K):
                step_strong(W + i)
            dec_s.wait(stream.cuda_stream)
            e1.record(stream)
        barrier()
        ms_s = max_over_ranks(e0.elapsed_time(e1))
        strong = {"value": world * Ss * BLK * K / (ms_s * 1e-3) / 1e6, "unit": "MS/s", "ms_per_step": ms_s / K,
                  "streams_total": world * Ss, "streams_per_gpu": Ss, "scaling": "strong",
                  "note": "fewer streams per GPU starve the lane-per-stream kernels (their time does not depend on the "
                          "stream count): DESIGN.md section 5"}
        dec_s.close()
    elif not args.no_extras:
        strong = {"value": value, "unit": "MS/s", "ms_per_step": ms / K, "streams_total": S, "streams_per_gpu": S,
                  "scaling": "strong", "note": "N = 1: identical to the weak-scaling figure"}

    # ---- tolerance mode (rfm_config::fir_fused = 1, opt-in; VERDICT r01 item 7): the same device-resident steps with
    # fused multiply-adds in the FIRs, and how far the audio moves from the exact mode's on the same blocks
    tol = None
    if not args.no_extras:
        dec_t = rfm.FmDecoderBatch(FS, -0.15 * FS, downsample=DS, n_streams=S, max_block_len=BLK, device=local,
                                   lanes_sms=args.lanes_sms, fir_fused=1)
        dec_x = rfm.FmDecoderBatch(FS, -0.15 * FS, downsample=DS, n_streams=S, max_block_len=BLK, device=local,
                                   lanes_sms=args.lanes_sms)
        audio_t = torch.zeros_like(audio)
        err, err_sum, err_dif = 0.0, 0.0, 0.0
        nchk = 20
        with torch.cuda.stream(stream):
            for i in range(max(W, nchk)):
                k_t = dec_t.process_u8_device(iq.data_ptr() + (i % nres) * BLK * esz, nres * BLK, BLK, audio_t.data_ptr(), stride,
                                              stream.cuda_stream)
                dec_t.wait(stream.cuda_stream)
                if i < nchk:
                    dec_x.process_u8_device(iq.data_ptr() + (i % nres) * BLK * esz, nres * BLK, BLK, audio.data_ptr(), stride,
                                            stream.cuda_stream)
                    dec_x.wait(stream.cuda_stream)
                    a_t, a_x = audio_t[:, :k_t].double().view(S, -1, 2), audio[:, :k_t].double().view(S, -1, 2)
                    err = max(err, float((a_t - a_x).abs().max()))
                    err_sum = max(err_sum, float((a_t.sum(-1) - a_x.sum(-1)).abs().max()))
                    err_dif = max(err_dif, float(((a_t[..., 0] - a_t[..., 1]) - (a_x[..., 0] - a_x[..., 1])).abs().max()))
        dec_x.close()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for i in range(K):
                dec_t.process_u8_device(iq.data_ptr() + ((W + i) % nres) * BLK * esz, nres * BLK, BLK, audio_t.data_ptr(), stride,
                                        stream.cuda_stream)
            dec_t.wait(stream.cuda_stream)
            e1.record(stream)
        barrier()
        ms_t = max_over_ranks(e0.elapsed_time(e1))
        dec_t.close()
        tol = {"config": "rfm_config::fir_fused = 1 (FFMA in the front-end FIR, the resamplers and the rotating FIRs; every PLL / "
                         "IIR / conversion unchanged)", "value": world * S * BLK * K / (ms_t * 1e-3) / 1e6, "unit": "MS/s",
               "ms_per_step": ms_t / K, "max_abs_audio_diff_vs_exact": err, "max_abs_LplusR_diff": err_sum,
               "max_abs_LminusR_diff": err_dif, "blocks_compared": nchk, "streams_compared": S,
               "note": "not the headline: the default (and every parity test) is the bit-exact mode"}

    c5 = c5_leg(torch, rfm, rank, world, local, barrier, max_over_ranks) if not args.no_extras else None
    single = single_stream_leg(rfm, local) if (rank == 0 and not args.no_extras) else None
    cpu = cpu_baseline_leg() if (rank == 0 and world == 1 and not args.no_cpu) else None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": workload_config(world), "roofline": roofline,
                "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clk,
                "audio_floats_per_stream_per_step": nfl,
                "demod_chunks_repaired": repairs, "host_enqueue_ms_per_step": host_enqueue_ms,
                "strong": strong, "c5": c5, "single_stream": single, "tolerance_mode": tol}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=STREAMS_PER_GPU)
    ap.add_argument("--groups", type=int, default=0)
    ap.add_argument("--host-groups", type=int, default=4,
                    help="stream groups of the host-buffer (e2e) decoder: 4 measured best for 4096 streams -- blocking call 12.0 ms "
                         "(8 groups: 14.3, 1 group: 13.9), streaming 10.2 ms (profiles/r02_e2e_host_groups.txt)")
    ap.add_argument("--resident-blocks", type=int, default=12)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-prof", action="store_true", help="do not bracket kernels with CUDA events (roofline leg off)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling / C5 / single-stream legs")
    ap.add_argument("--lanes-sms", type=int, default=0, help="rfm_config::lanes_sms (0 = automatic, 1 = no SM partition)")
    ap.add_argument("--fir-fused", type=int, default=0, help="rfm_config::fir_fused for the main legs (1 = tolerance mode; the "
                                                             "headline is the default 0)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the audio of the last timed step and the RDS groups "
                                                          "decoded by then as DIR/*.npy (at most 64 MB; see dump_outputs), "
                                                          "to compare two builds output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
