#!/usr/bin/env python
"""Throughput of the IQ sample chain FreqShifter -> Filter -> Downsampler on B200.

    python bench.py --gpus N --steps K --warmup W            # CUDA arm (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm (the reference's algorithm on host cores)
    python bench.py --steps K --dump-outputs DIR             # + the last timed step's outputs as DIR/*.npy

Workload (BASELINE.json configs[2], the one the metric's "1/2/4/8 B200" sharding
is defined on): a channelizer batch of independent 2.4 MS/s complex-f32
streams, each FreqShifter(per-stream shift) -> Filter(3 kHz low-pass, n = 4096)
-> Downsampler(48 kS/s, bandwidth 6 kHz).  One step = one push of
CHUNKS_PER_STEP chunks for every stream.  Streams are sharded over ranks with no
data-path collective (weak scaling: STREAMS_PER_GPU per rank).

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMPLE_RATE = 2_400_000.0
CHUNK_LEN = 4096
OUT_RATE = 48_000.0
BANDWIDTH = 6_000.0
CUTOFF = 3_000.0
OUT_CHUNK = 2048
BYTES_PER_SAMPLE = 8.0 * (1.0 + OUT_RATE / SAMPLE_RATE)  # SURVEY.md 8(d): read once + written once
METRIC = "complex MS/s via FreqShift->Filter->Downsampler"
UNIT = "MS/s"
# --dump-outputs writes at most this many bytes: a seeded sample of the streams when one step's output is larger
# (4096 streams x 4096 complex64 samples = 128 MB at the default size)
DUMP_BYTES = 32 << 20




def ncu_traffic(kernel: str, streams: int, chunks: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel` from the `ncu --set full` capture of this
    very command, recorded with the commit it was taken at in profiles/ncu_traffic.json (written by
    profiles/ncu_summary.py).  None when no capture of this kernel / shape is on record."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    try:
        with open(p) as fh:
            d = json.load(fh)
    except Exception:
        return None, None
    e = d.get(f"{kernel}:{streams}x{chunks}")
    return (e["dram_bytes_per_launch"], e) if e else (None, None)


def stream_shift(stream_id: int) -> float:
    """SURVEY.md 8(d), config C3."""
    return float((stream_id * 577) % 2_400_000 - 1_200_000)


def lowpass(cutoff):
    def f(_bin, freq):
        return 1.0 + 0.0j if abs(freq) <= cutoff else 0.0j

    return f


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "10", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self, name):
        """wall-clock bracket of the timed region: only samples inside it are reported"""
        setattr(self, name, time.time())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t0, t1 = getattr(self, "t0", None), getattr(self, "t1", None)
        inside = [ln for ts, ln in self.lines if t0 is not None and t1 is not None and t0 <= ts <= t1 + 0.02]
        scope = "timed region" if inside else "around the timed region"
        for ln in (inside or [ln for _, ln in self.lines]):
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(max(mx)) if mx else None,
            "samples": len(sm),
            "scope": scope,
            "reasons": sorted(reasons),
        }


# ---------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle restatement) on the host cores
# ---------------------------------------------------------------------------
_CPU_INPUT = {}


def cpu_chain_run(cores: int, streams_per_core: int, n_chunks: int):
    """Times the oracle's C restatement of the reference loops (oracle/radiorust_oracle.c) on `cores` threads over
    independent streams; returns (MS/s, seconds, description of what was timed, seconds spent on the phase tables).
    The FreqShifter phase tables (transform.rs:321-340: built once per retune) are built BEFORE the timed call."""
    from oracle import oracle_c
    from oracle import radiorust_oracle as orc

    S = cores * streams_per_core
    key = (S, n_chunks)
    if key not in _CPU_INPUT:  # synthetic input of the sample: generated once, reused by every step
        base = orc.synth_noise(20260000 + 3 * 100000, n_chunks * CHUNK_LEN, "f32")
        _CPU_INPUT.clear()
        _CPU_INPUT[key] = np.stack([np.roll(base, 977 * s) for s in range(S)])
        kw0 = dict(shifts=[stream_shift(s) for s in range(cores)], freq_resp=orc.lowpass(CUTOFF), down=(OUT_RATE, BANDWIDTH, 3.0),
                   n_threads=cores)
        oracle_c.chain(_CPU_INPUT[key][:cores, : 2 * CHUNK_LEN], "f32", SAMPLE_RATE, CHUNK_LEN, **kw0)  # warm up
    x = _CPU_INPUT[key]
    shifts = [stream_shift(s) for s in range(S)]
    kw = dict(shifts=shifts, freq_resp=orc.lowpass(CUTOFF), down=(OUT_RATE, BANDWIDTH, 3.0), n_threads=cores)
    t = {}
    oracle_c.chain(x, "f32", SAMPLE_RATE, CHUNK_LEN, timing=t, prebuilt_phase_tables=True, **kw)
    dt = t["seconds"]
    samples = S * n_chunks * CHUNK_LEN
    desc = (f"{S} streams x {n_chunks} chunks x {CHUNK_LEN} samples of the same chain (per-stream shifts, 3 kHz Filter, Downsampler to "
            f"48 kS/s) on {cores} pthreads over streams: C restatement of the reference loops (oracle/radiorust_oracle.c, gcc -O3 with "
            f"AVX-512/AVX2 clones; radix-4 Stockham FFT standing in for rustfft; two 8192-point FFTs per chunk like filters.rs:244-252). "
            f"Timed: the per-chunk hot loops; NOT timed: filter/tap design and the FreqShifter phase tables "
            f"({t.get('table_seconds', 0.0):.2f} s for this sample), which the reference builds once per retune")
    return samples / dt / 1e6, dt, desc, t.get("table_seconds", 0.0)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


REF_STREAMS_PER_CORE = 2
REF_CHUNKS = 1000


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    vals = []
    for i in range(args.warmup + args.steps):
        v, dt, desc, tab = cpu_chain_run(cores, REF_STREAMS_PER_CORE, REF_CHUNKS)
        if i >= args.warmup:
            vals.append((v, dt))
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals])) * 1e3
    cfg = workload_config(args, 1)
    # what this arm actually timed per step (a bounded sample of the workload above, on the host cores)
    cfg["reference_sample"] = {"streams": cores * REF_STREAMS_PER_CORE, "chunks_per_step": REF_CHUNKS, "chunk_len": CHUNK_LEN,
                               "samples_per_step": cores * REF_STREAMS_PER_CORE * REF_CHUNKS * CHUNK_LEN, "threads": cores}
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {
        "workload": "configs[2] channelizer batch: independent 2.4 MS/s complex-f32 streams, FreqShifter(per-stream shift) -> "
                    "Filter(3 kHz low-pass, n=4096, N=8192) -> Downsampler(48 kS/s, bw 6 kHz, L=343)",
        "streams_per_gpu": args.streams, "streams_total": args.streams * world, "chunk_len": CHUNK_LEN,
        "chunks_per_step": args.chunks, "sample_rate": SAMPLE_RATE, "output_rate": OUT_RATE,
        "l2_policy": "inputs larger than L2 (%.2f GB per step per GPU), no flush" % (args.streams * args.chunks * CHUNK_LEN * 8 / 1e9),
        "sharding": "streams block-partitioned over ranks, no collective on the data path",
    }


def bind_to_gpu_cpus(index):
    """Keep this rank's threads (and, by first touch, its pinned host buffers) on the CPUs next to its GPU, as a
    multi-GPU host application would: eight ranks copying from one NUMA node share that node's memory bandwidth.
    Returns the number of CPUs bound to, or None when NVML / the affinity call is not available."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None



# ---------------------------------------------------------------------------
# CUDA arm helpers
# ---------------------------------------------------------------------------
def _time_pushes(torch, chain, sr, n, chunks, x_ptr, in_stride, y_ptr, cap, steps, warmup):
    """ms per push of `steps` back-to-back device-resident pushes (CUDA events on the chain's stream)."""
    ext = torch.cuda.ExternalStream(chain.cuda_stream)
    for _ in range(warmup):
        chain.push_device(sr, n, chunks, x_ptr, in_stride, y_ptr, cap, cap)
    chain.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ext):
        e0.record(ext)
        for _ in range(steps):
            chain.push_device(sr, n, chunks, x_ptr, in_stride, y_ptr, cap, cap)
        e1.record(ext)
    chain.sync()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def dump_outputs(out_dir, torch, y, count):
    """Writes what the last timed push returned to its caller, y[s, :count] per stream (complex64 as float32 pairs), for
    a fixed, seeded sample of the streams that keeps the files within DUMP_BYTES: out_dir/output.npy [streams, count, 2]
    float32, and the sampled stream indices as out_dir/output_streams.npy (float64)."""
    S = y.shape[0]
    k = min(S, max(1, DUMP_BYTES // max(8 * count, 1)))
    n = min(count, DUMP_BYTES // (8 * k))
    ids = np.sort(np.random.default_rng(20260000).choice(S, size=k, replace=False))
    sample = y[torch.from_numpy(ids).to(y.device), :n].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output.npy"), sample)
    np.save(os.path.join(out_dir, "output_streams.npy"), ids.astype(np.float64))


def _spot_check(rr, ctx, stages, ostages, flt, sr, n, chunks, x_host):
    """relative L2 error of the CUDA chain against the oracle on one small host-side stream (the parity spot check that
    goes with every configuration's throughput figure)"""
    from oracle import radiorust_oracle as orc

    ch = rr.Chain(ctx, stages, flt, n_streams=1)
    parts = []
    half = max(1, chunks // 2)
    for lo, hi in ((0, half), (half, chunks)):
        if hi > lo:
            y, _ = ch.push(sr, np.ascontiguousarray(x_host[lo * n:hi * n]), n)
            parts.append(y[0].copy())
    plan = ch.plan
    ch.close()
    got = np.concatenate(parts)
    want = orc.Chain(ostages()).run(sr, x_host[: chunks * n], n)
    if got.shape != want.shape or want.size == 0:
        return None, plan
    return orc.rel_l2(got, want), plan


def other_configs(torch, rr, ctx, peak):
    """The other BASELINE.json configs on one B200, outside the headline's timed region: device-resident throughput
    (input samples per second), its HBM-roofline fraction on SURVEY.md 8d's bytes per input sample, the plan, and a
    parity spot check against the oracle.  Streams are batched where the config is a single stream (replicas)."""
    from oracle import radiorust_oracle as orc  # the checker of the parity spot checks, never the thing measured

    out = {}

    def deemph_resp(tau):
        def f(bin_, freq):  # examples/relm_app/simple_receiver.rs:43-49 with filters.rs:20-27
            if bin_ != 0 and 20.0 <= abs(freq) <= 16000.0:
                return 1.0 / complex(1.0, 2.0 * np.pi * tau * freq)
            return 0j

        return f

    def lp(c):
        return lowpass(c)

    def run(name, flt, sr, n, S, chunks, stages, bytes_per_sample, spot, steps=5, warmup=2):
        cdt = torch.float32 if flt == "f32" else torch.float64
        gen = torch.Generator(device="cuda")
        gen.manual_seed(20260000 + len(out))
        x = torch.randn((S, chunks * n, 2), device="cuda", dtype=cdt, generator=gen)
        chain = rr.Chain(ctx, stages, flt, n_streams=S)
        cap = chain.max_output(sr, n, chunks + 2) + 8192
        y = torch.zeros((S, cap, 2), device="cuda", dtype=cdt)
        chain.push_device(sr, n, chunks, x.data_ptr(), chunks * n, y.data_ptr(), cap, cap)  # start-up chunks (stateful path)
        ms = _time_pushes(torch, chain, sr, n, chunks, x.data_ptr(), chunks * n, y.data_ptr(), cap, steps, warmup)
        plan = chain.plan
        chain.close()
        del x, y
        torch.cuda.empty_cache()
        value = S * chunks * n / (ms * 1e-3) / 1e6
        err, plan_small = spot()
        out[name] = {"value": value, "unit": UNIT, "ms_per_push": ms, "streams": S, "chunks_per_push": chunks, "chunk_len": n,
                     "dtype": flt, "plan": plan, "bytes_per_input_sample": bytes_per_sample,
                     "roofline": {"bound": "hbm", "achieved": value * 1e6 * bytes_per_sample / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": value * 1e6 * bytes_per_sample / 1e9 / peak},
                     "rel_l2": err, "rel_l2_tolerance": 1e-5 if flt == "f32" else 1e-12, "spot_check_plan": plan_small}

    # C1: 1.024 MS/s -> 48 kS/s, n = 4096, P/Q = 64/3, batched
    sr, n = 1_024_000.0, 4096
    st = [rr.FreqShifter(123457.0), rr.Filter.new(lp(3000.0)), rr.Downsampler(192, 48000.0, 6000.0)]
    run("C1_batched", "f32", sr, n, 4096, 48, st, 8.0 * (1 + 48000.0 / sr),
        lambda: _spot_check(rr, ctx, st, lambda: [orc.FreqShifter("f32", 1.0, 123457.0), orc.Filter.new("f32", orc.lowpass(3000.0)),
                                                  orc.Downsampler("f32", 192, 48000.0, 6000.0)], "f32", sr, n, 12,
                            orc.synth_noise(20260000 + 100000, 12 * n, "f32")))
    # C2: one 20 MS/s stream, n = 65536, Downsampler L = 2858 (64 replicas)
    sr, n = 20_000_000.0, 65536
    st2 = [rr.FreqShifter(1_234_567.0), rr.Filter.new(lp(3000.0)), rr.Downsampler(128, 48000.0, 6000.0)]
    run("C2_batched", "f32", sr, n, 64, 16, st2, 8.0 * (1 + 48000.0 / sr),
        lambda: _spot_check(rr, ctx, st2, lambda: [orc.FreqShifter("f32", 1.0, 1_234_567.0), orc.Filter.new("f32", orc.lowpass(3000.0)),
                                                   orc.Downsampler("f32", 128, 48000.0, 6000.0)], "f32", sr, n, 5,
                            orc.synth_noise(20260000 + 200000, 5 * n, "f32")))
    # ... and 256 replicas: the front end's 128-row tiles come in whole waves of CTAs only with more streams (64 x 7 tiles
    # = 448 CTAs on 296 resident ones is two rounds, the second half empty)
    run("C2_batched_256", "f32", sr, n, 256, 16, st2, 8.0 * (1 + 48000.0 / sr), lambda: (out["C2_batched"]["rel_l2"], out["C2_batched"]["spot_check_plan"]))
    # C4: 256 FM stations at 10 MS/s, Filter -> FmDemod -> de-emphasis -> Downsampler(48 kS/s), L = 7500
    sr, n = 10_000_000.0, 65536
    de = deemph_resp(50e-6)
    st4 = [rr.Filter.new(lp(100000.0)), rr.FmDemod(75000.0), rr.Filter.new_rectangular(de), rr.Downsampler(4096, 48000.0, 40000.0)]
    st4s = [rr.Filter.new(lp(100000.0)), rr.FmDemod(75000.0), rr.Filter.new_rectangular(de), rr.Downsampler(64, 48000.0, 40000.0)]
    run("C4_fm_256_stations", "f32", sr, n, 256, 8, st4, 8.0 * (1 + 48000.0 / sr),
        lambda: _spot_check(rr, ctx, st4s, lambda: [orc.Filter.new("f32", orc.lowpass(100000.0)), orc.FmDemod("f32", 75000.0),
                                                    orc.Filter.new_rectangular("f32", de), orc.Downsampler("f32", 64, 48000.0, 40000.0)],
                            "f32", sr, n, 6, orc.synth_fm_station(20260000 + 400000, 6 * n, sr, 75000.0, 15000.0, -30.0, "f32")))
    # C5: f64 Filter with a 2^20-point FFT
    sr, n = 2_400_000.0, 1 << 19
    st5 = [rr.Filter.new(lp(20000.0))]
    run("C5_filter_f64_2pow20", "f64", sr, n, 16, 4, st5, 32.0,
        lambda: _spot_check(rr, ctx, st5, lambda: [orc.Filter.new("f64", orc.lowpass(20000.0))], "f64", sr, n, 3,
                            orc.synth_noise(20260000 + 500000, 3 * n, "f64")))
    # C5: f64 Upsampler 48 kS/s -> 2.4 MS/s, L = 515
    sr, n = 48000.0, 4096
    st5u = [rr.Upsampler(4096, 2_400_000.0, 20000.0)]
    run("C5_upsampler_f64", "f64", sr, n, 64, 8, st5u, 16.0 * (1 + 50.0),
        lambda: _spot_check(rr, ctx, st5u, lambda: [orc.Upsampler("f64", 4096, 2_400_000.0, 20000.0)], "f64", sr, 1024, 3,
                            orc.synth_noise(20260000 + 500001, 3 * 1024, "f64")))
    return out


# ---------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------
def run_cuda(args):
    import torch
    import radiorust_b200 as rr

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_cpus(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")  # the gather runs under the next push's kernels
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    S, C_ = args.streams, args.chunks
    length = C_ * CHUNK_LEN
    ctx = rr.Context(local)
    stages = [rr.FreqShifter(0.0), rr.Filter.new(lowpass(CUTOFF)), rr.Downsampler(OUT_CHUNK, OUT_RATE, BANDWIDTH)]
    chain = rr.Chain(ctx, stages, "f32", n_streams=S)
    from radiorust_b200 import sharding

    g_lo, g_hi = sharding.weak_scaling_streams(rank, world, S)  # global stream ids of this rank (weak scaling)
    chain.set_shifts(0, [stream_shift(g) for g in range(g_lo, g_hi)])

    gen = torch.Generator(device="cuda")
    gen.manual_seed(20260000 + 3 * 100000 + rank)
    x = torch.randn((S, length, 2), device="cuda", dtype=torch.float32, generator=gen)
    cap = chain.max_output(SAMPLE_RATE, CHUNK_LEN, C_ + 1) + OUT_CHUNK
    y = torch.zeros((S, cap, 2), device="cuda", dtype=torch.float32)
    torch.cuda.synchronize()

    ext = torch.cuda.ExternalStream(chain.cuda_stream)

    def step():
        return chain.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y.data_ptr(), cap, cap)

    for _ in range(args.warmup):
        step()
    chain.sync()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    launches0 = rr.kernel_launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    chain.set_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out_total = 0
    if rank == 0:
        time.sleep(0.05)  # let the sampler come up
        sampler.mark("t0")
    with torch.cuda.stream(ext):
        e0.record(ext)
        for _ in range(args.steps):
            cnt, _rate = step()
            out_total += cnt
        e1.record(ext)
    chain.sync()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.mark("t1")
    if dist is not None:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = rr.kernel_launch_count() - launches0
    elapsed_ms = e0.elapsed_time(e1)
    k_ms, k_n, k_name = chain.kernel_time()
    k_all = chain.kernel_breakdown()
    chain.set_timing(False)
    plan = chain.plan
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, y, cnt)  # before anything else writes y
    if dist is not None:
        t = torch.tensor([elapsed_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    samples_step = S * length
    value = samples_step * world * args.steps / (elapsed_ms * 1e-3) / 1e6

    # ---- the one collective of the path: gathering the channelizer outputs (SURVEY 8e) --------------
    # Outside the timed region and reported separately.  (a) NCCL all-gather of one step's decimated samples, alone, for
    # reference.  (b) The product's way: every rank's chain stores its outputs straight into rank 0's buffer over NVLink
    # (the buffer is opened through CUDA IPC and passed as dev_out, so the last kernel's epilogue does the transfer: no
    # collective kernel competes with the persistent k_fused CTAs for SMs); the steps are timed again with that destination.
    gather = None
    strong = None
    if dist is not None:
        import ctypes as C

        from radiorust_b200 import _ffi

        lib = _ffi.load()
        per_stream = out_total // max(args.steps, 1)
        mine = y[:, :per_stream].contiguous()
        everyone = torch.empty((world * S, per_stream, 2), device="cuda", dtype=torch.float32)
        dist.all_gather_into_tensor(everyone, mine)  # warm-up (communicator set-up)
        torch.cuda.synchronize()
        dist.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        g0.record()
        for _ in range(reps):
            dist.all_gather_into_tensor(everyone, mine)
        g1.record()
        torch.cuda.synchronize()
        t = torch.tensor([g0.elapsed_time(g1) / reps], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gms = float(t.item())
        gather = {"nccl_all_gather_alone": {"ms": gms, "bytes_per_rank": mine.numel() * 4, "bytes_total": everyone.numel() * 4,
                                            "share_of_step": gms / (elapsed_ms / args.steps)}}
        del everyone, mine

        # (b) gather-to-root fused into the chain's last kernel: rank 0 owns [world*S][cap] complex64
        root_bytes = world * S * cap * 8
        root_ptr = C.c_void_p()
        handle = (C.c_ubyte * 64)()
        if rank == 0:
            _ffi.check(lib.rr_device_alloc(ctx._h, root_bytes, C.byref(root_ptr)))
            _ffi.check(lib.rr_ipc_export(ctx._h, root_ptr, handle))
        obj = [bytes(handle)]
        dist.broadcast_object_list(obj, src=0)
        if rank != 0:
            hb = (C.c_ubyte * 64).from_buffer_copy(obj[0])
            _ffi.check(lib.rr_ipc_open(ctx._h, hb, C.byref(root_ptr)))
        my_out = root_ptr.value + rank * S * cap * 8
        # two chains in lock step: one stores into rank 0's buffer, the twin locally (to check what arrived)
        ch_p2p = rr.Chain(ctx, stages, "f32", n_streams=S)
        ch_loc = rr.Chain(ctx, stages, "f32", n_streams=S)
        for chx in (ch_p2p, ch_loc):
            chx.set_shifts(0, [stream_shift(g) for g in range(g_lo, g_hi)])
        y_loc = torch.zeros((S, cap, 2), device="cuda", dtype=torch.float32)
        for _ in range(3):
            ch_p2p.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, my_out, cap, cap)
            ch_loc.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y_loc.data_ptr(), cap, cap)
        ch_p2p.sync()
        ch_loc.sync()
        torch.cuda.synchronize()
        dist.barrier()
        ms_loc = _time_pushes(torch, ch_loc, SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y_loc.data_ptr(), cap, args.steps, 0)
        dist.barrier()
        ms_p2p = _time_pushes(torch, ch_p2p, SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, my_out, cap, args.steps, 0)
        t = torch.tensor([ms_loc, ms_p2p], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_loc, ms_p2p = float(t[0].item()), float(t[1].item())
        # both chains have now seen the same pushes: their last outputs must agree, bit for bit, on rank 0's side
        cnt_p, _ = ch_p2p.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, my_out, cap, cap)
        cnt_l, _ = ch_loc.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y_loc.data_ptr(), cap, cap)
        ch_p2p.sync()
        ch_loc.sync()
        torch.cuda.synchronize()
        dist.barrier()
        sums = [None] * world
        dist.all_gather_object(sums, (int(cnt_l), float(y_loc[:, :cnt_l].double().abs().sum().item())))
        intact = None
        if rank == 0:
            host = np.empty((world * S, cap, 2), dtype=np.float32)
            _ffi.check(lib.rr_memcpy_d2h(ctx._h, host.ctypes.data_as(C.c_void_p), root_ptr, root_bytes))  # (waits for the device)
            intact = all(abs(float(np.abs(host[r * S:(r + 1) * S, :sums[r][0]].astype(np.float64)).sum()) - sums[r][1]) <= 1e-9 * max(1.0, sums[r][1])
                         for r in range(world))
            del host
        dist.barrier()
        # (c) the same gather by copy engine: outputs stay local (two buffers), and a device-to-device copy on the chain's
        # copy stream moves each push's outputs into rank 0's buffer while the next push computes
        ys2 = [y_loc, torch.zeros_like(y_loc)]
        ch_ce = rr.Chain(ctx, stages, "f32", n_streams=S)
        ch_ce.set_shifts(0, [stream_shift(g) for g in range(g_lo, g_hi)])

        def ce_steps(k):
            ext2 = torch.cuda.ExternalStream(ch_ce.cuda_stream)
            e_a, e_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(ext2):
                e_a.record(ext2)
            last = 0
            for i in range(k):
                yy = ys2[i & 1]
                cnt_i, _ = ch_ce.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, yy.data_ptr(), cap, cap)
                ch_ce.copy_out_async(my_out, cap, yy.data_ptr(), cap, cnt_i)
                last = cnt_i
            with torch.cuda.stream(ext2):
                e_b.record(ext2)
            t0 = time.perf_counter()
            ch_ce.sync()
            torch.cuda.synchronize()
            return e_a.elapsed_time(e_b) / k, last

        for _ in range(2):
            ce_steps(2)
        dist.barrier()
        t_w0 = time.perf_counter()
        ms_ce_dev, cnt_ce = ce_steps(args.steps)
        ms_ce = (time.perf_counter() - t_w0) * 1e3 / args.steps  # host clock: includes the last copy
        t = torch.tensor([ms_ce, ms_ce_dev], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_ce, ms_ce_dev = float(t[0].item()), float(t[1].item())
        ch_ce.close()
        gather["copy_engine_into_root"] = {
            "what": "outputs stay local (two buffers); rr_chain_copy_out_async moves each push's outputs into rank 0's buffer on the "
                    "chain's copy stream (copy engine over NVLink) under the next push's kernels",
            "ms_per_step": ms_ce, "ms_per_step_kernels_only": ms_ce_dev, "ms_per_step_local_output": ms_loc,
            "overhead_frac": ms_ce / ms_loc - 1.0, "value": S * length * world / (ms_ce * 1e-3) / 1e6, "unit": UNIT,
        }
        del ys2
        gather["p2p_store_into_root"] = {
            "what": "every rank's last kernel stores its outputs into rank 0's buffer (CUDA IPC mapping, NVLink peer stores)",
            "ms_per_step": ms_p2p, "ms_per_step_local_output": ms_loc, "overhead_frac": ms_p2p / ms_loc - 1.0,
            "value": S * length * world / (ms_p2p * 1e-3) / 1e6, "unit": UNIT, "root_copy_matches_every_rank": intact,
            "bytes_per_step_into_root": int(sum(c for c, _ in sums)) * S * 8,
        }
        ch_p2p.close()
        ch_loc.close()
        if rank != 0:
            lib.rr_ipc_close(ctx._h, root_ptr)
        dist.barrier()
        if rank == 0:
            lib.rr_device_free(ctx._h, root_ptr)

        # ---- strong scaling: configs[2]'s 4096 streams in total, sharded over the ranks ------------------------
        s_lo, s_hi = sharding.stream_range(rank, world, args.streams)  # block partition of the 4096 streams
        S_str = s_hi - s_lo
        if args.streams >= world:
            ch_s = rr.Chain(ctx, stages, "f32", n_streams=S_str)
            ch_s.set_shifts(0, [stream_shift(g) for g in range(s_lo, s_hi)])
            ch_s.push_device(SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y.data_ptr(), cap, cap)
            dist.barrier()
            ms_s = _time_pushes(torch, ch_s, SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y.data_ptr(), cap, args.steps, 3)
            t = torch.tensor([ms_s], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_s = float(t.item())
            strong = {"scaling": "strong", "streams_total": args.streams, "streams_per_gpu": S_str, "ms_per_step": ms_s,
                      "value": sharding.aggregate_throughput(args.streams * length, 1, ms_s * 1e-3) / 1e6, "unit": UNIT, "plan": ch_s.plan}
            ch_s.close()

    # ---- end to end: pinned host chunks in, host result out, through rr_chain_push ----
    e2e = None
    if not args.no_e2e:
        e_steps = max(1, min(args.steps, args.e2e_steps))
        hx = torch.empty((S, length, 2), dtype=torch.float32, pin_memory=True)
        blk = torch.randn((min(S, 64), length, 2), dtype=torch.float32)
        for s0 in range(0, S, blk.shape[0]):
            hx[s0 : s0 + blk.shape[0]] = blk[: min(blk.shape[0], S - s0)]
        hy = torch.empty((S, cap, 2), dtype=torch.float32, pin_memory=True)

        hy2 = torch.empty((S, cap, 2), dtype=torch.float32, pin_memory=True)
        outs = [hy, hy2]

        def estep(i):
            # no sync between pushes: the library's two staging slots overlap the H2D copy of push i+1 with the kernels
            # and the D2H copy of push i (rr_chain_push); the host reads a result only after rr_chain_sync
            cnt, _ = chain.push_host_async(SAMPLE_RATE, CHUNK_LEN, C_, hx.data_ptr(), length, outs[i & 1].data_ptr(), cap, cap)
            return cnt

        estep(0)  # warm-up: both staging slots of the library get their buffers outside the timed region
        estep(1)
        chain.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        d2h = 0
        t_e0 = time.perf_counter()
        for i in range(e_steps):
            d2h += estep(i) * S * 8
        chain.sync()
        torch.cuda.synchronize()
        ems = (time.perf_counter() - t_e0) * 1e3  # host clock around enqueue .. last result on the host (copies on 3 streams)
        float(hy[0, 0, 0])  # the device->host read of the result
        if dist is not None:
            t = torch.tensor([ems], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        e2e = {
            "value": samples_step * world * e_steps / (ems * 1e-3) / 1e6, "unit": UNIT,
            "h2d_bytes_per_step": samples_step * 8, "d2h_bytes_per_step": d2h // e_steps, "steps": e_steps,
            "api": "rr_chain_push (pinned host chunks -> H2D -> kernels -> D2H), per rank; pushes back to back, one sync at the end",
            "cpus_bound_per_rank": numa,
        }
        del hx, hy, hy2

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_kind = measured_peaks()
    extras = {}
    if world == 1 and not args.no_extras:
        # ---- push size: the block API delivers one chunk per message; how throughput depends on chunks per push ----
        sweep = {}
        for cpp in (1, 8, 50):
            if cpp > C_:
                continue
            ms = _time_pushes(torch, chain, SAMPLE_RATE, CHUNK_LEN, cpp, x.data_ptr(), length, y.data_ptr(), cap, 20, 5)
            v = S * cpp * CHUNK_LEN / (ms * 1e-3) / 1e6
            sweep[str(cpp)] = {"ms_per_push": ms, "value": v, "unit": UNIT, "plan": chain.plan,
                               "step_frac": v * 1e6 * BYTES_PER_SAMPLE / 1e9 / peak}
        extras["push_size_sweep"] = sweep
        # ---- sustained: the same steps back to back for >= 2 s (the board reaches its power cap) -------------------
        per = elapsed_ms / args.steps
        n_sus = int(max(50, min(20000, 2200.0 / max(per, 1e-3))))
        smp = ClockSampler(local)
        smp.start()
        time.sleep(0.05)
        smp.mark("t0")
        ms = _time_pushes(torch, chain, SAMPLE_RATE, CHUNK_LEN, C_, x.data_ptr(), length, y.data_ptr(), cap, n_sus, 0)
        smp.mark("t1")
        v = S * length / (ms * 1e-3) / 1e6
        extras["sustained"] = {"steps": n_sus, "seconds": ms * n_sus / 1e3, "ms_per_step": ms, "value": v, "unit": UNIT,
                               "step_frac": v * 1e6 * BYTES_PER_SAMPLE / 1e9 / peak, "clocks": smp.stop()}
    traffic, traffic_rec = ncu_traffic(k_name, S, C_)
    if args.traffic is not None:
        traffic, traffic_rec = args.traffic, {"source": "--traffic"}
    k_avg_ms = k_ms / max(k_n, 1)
    achieved = samples_step * BYTES_PER_SAMPLE / (k_avg_ms * 1e-3) / 1e9 if k_n else None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (torch.randn on device, seeded)",
        "config": workload_config(args, world),
        "plan": plan,
        "clocks": clocks,
        "e2e": e2e,
        "gather": gather,
        "gpu_launches": int(launches),
        "roofline": {
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
            "traffic": traffic, "traffic_record": traffic_rec, "peak_kind": peak_kind, "kernel": k_name, "kernel_ms": k_avg_ms, "kernel_launches": k_n,
            "algorithmic_bytes_per_launch": samples_step * BYTES_PER_SAMPLE,
            "kernel_share_of_step": (k_ms / elapsed_ms) if elapsed_ms else None,
            "kernels": {nm: {"ms_per_launch": ms / max(n, 1), "launches": n, "share_of_step": ms / elapsed_ms}
                        for nm, (ms, n) in k_all.items()},
            # the same algorithmic bytes over the whole step (all kernels of a push), for comparison
            "step_achieved": value * 1e6 * BYTES_PER_SAMPLE / world / 1e9, "step_frac": value * 1e6 * BYTES_PER_SAMPLE / world / 1e9 / peak,
        },
        "output_samples_per_step": out_total // max(args.steps, 1),
    }
    line.update(extras)
    if strong is not None:
        line["strong_scaling"] = strong
    if world == 1 and not args.no_extras:
        # the big buffers of the headline go first: the other configs bring their own
        chain.close()
        del x, y
        torch.cuda.empty_cache()
        try:
            line["configs"] = other_configs(torch, rr, ctx, peak)
        except Exception as e:  # the headline line must not be lost to a side measurement
            line["configs"] = {"error": repr(e)}
    if world == 1 and not args.no_cpu:
        cores = host_cores()
        v, dt, desc, tab = cpu_chain_run(cores, REF_STREAMS_PER_CORE, REF_CHUNKS)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc, "seconds": dt,
                                "phase_table_seconds_not_timed": tab}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="streams per GPU")
    ap.add_argument("--chunks", type=int, default=50, help="chunks per stream per step")
    ap.add_argument("--e2e-steps", type=int, default=6)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the push-size sweep, the sustained run and the other configs")
    ap.add_argument("--traffic", type=float, default=None, help="dram bytes per launch from an ncu --set full capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0, a seeded sample of its streams) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA arm")
    if args.warmup < 3 and args.impl == "cuda":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
