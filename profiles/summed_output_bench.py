#!/usr/bin/env python
"""Summed-output pushes of a transmit channelizer against per-stream pushes plus a sum over streams.

    python profiles/summed_output_bench.py --out r04_summed_output.json [--steps 10 --warmup 3 --rounds 3]

The chain is a TX channelizer: FmMod(5 kHz) -> Upsampler(2400, 2.4 MS/s, 20 kHz) (L = 515, x50) -> FreqShifter with
stream s at (577 s mod 2.4e6) - 1.2e6 Hz.  rr_chain_push_summed_device runs it as one kernel (k_synth) and writes one
row; the per-stream arm is rr_chain_push_device (k_fmmod, k_upsample_phase, k_freqshift into S full-rate rows) plus
torch.sum over the streams, run only where its S rows and the Upsampler's staging buffers fit in device memory.  The
host-fed arm times rr_chain_push_summed from pinned buffers.  Upsampler x3 -> FreqShifter is the generic route
(k_stream_sum), so each side of the route choice has a workload.

Arms of a case are timed in turn, `rounds` times, `steps` pushes each (device arms: CUDA events on the chain's stream
around every push and its sum, a sync after it; host arm: a host clock around back-to-back pushes ending in one
sync).  The JSON records ms/push (median and spread over all rounds), input GS/s (streams x input samples per push
over the push time), the algorithmic bytes each arm moves per push (from the shapes) over its time, the kernel
breakdown, the plans, and the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OUT_RATE = 2_400_000.0


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    line = (r.stdout.strip().splitlines() or [""])[0]
    parts = [p.strip() for p in line.split(",")]
    return {"name": parts[0] if parts else None, "power_limit": parts[1] if len(parts) > 1 else None}


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "n": len(v)}


def tx_chain(rr, ctx, S, generic=False):
    if generic:
        stages = [rr.Upsampler(2400, 48000.0, 7000.0), rr.FreqShifter(0.0)]
        nco, rate = 1, 48000.0
    else:
        stages = [rr.FmMod(5000.0), rr.Upsampler(2400, OUT_RATE, 20000.0), rr.FreqShifter(0.0)]
        nco, rate = 2, OUT_RATE
    ch = rr.Chain(ctx, stages, "f32", n_streams=S)
    ch.set_shifts(nco, [float((s * 577) % int(rate) - rate / 2) for s in range(S)])
    return ch


def breakdown(ch, step, k=3):
    ch.set_timing(True)
    for _ in range(k):
        step()
    ch.sync()
    ch.kernel_time()
    b = {name: {"ms_per_push": ms / k, "launches_per_push": cnt / k} for name, (ms, cnt) in ch.kernel_breakdown().items()}
    ch.set_timing(False)
    return b


def bytes_per_push(arm, S, L, M):
    """HBM bytes the algorithm needs per push (complex f32 = 8 bytes): summed reads the S inputs and writes one row;
    the per-stream arm also writes S upsampled rows, reads and writes them in the mixer and reads them in the sum."""
    if arm == "summed":
        return S * L * 8 + M * 8
    return S * L * 8 + S * M * 8 * 4 + M * 8


def device_case(torch, rr, ctx, S, L, steps, warmup, rounds, generic=False):
    sr = 16000.0 if generic else 48000.0
    gen = torch.Generator(device="cuda")
    gen.manual_seed(20264000 + S + L)
    x = torch.randn((S, L, 2), device="cuda", dtype=torch.float32, generator=gen)
    arms = {}
    su = tx_chain(rr, ctx, S, generic)
    M = su.max_output(sr, L, 1)
    row = torch.empty((M, 2), device="cuda", dtype=torch.float32)
    arms["summed"] = (su, lambda: su.push_summed_device(sr, L, 1, x.data_ptr(), L, row.data_ptr(), M))
    free, _ = torch.cuda.mem_get_info()
    per_stream_bytes = S * M * 8 * 5  # output rows + the Upsampler's two staging buffers (1.5 x each) + the sum
    rows = None
    if not generic and per_stream_bytes < 0.8 * free:
        ps = tx_chain(rr, ctx, S)
        rows = torch.empty((S, M, 2), device="cuda", dtype=torch.float32)
        row2 = torch.empty((M, 2), device="cuda", dtype=torch.float32)

        def per_stream():
            r = ps.push_device(sr, L, 1, x.data_ptr(), L, rows.data_ptr(), M, M)
            with torch.cuda.stream(torch.cuda.ExternalStream(ps.cuda_stream)):
                torch.sum(torch.view_as_complex(rows), dim=0, out=torch.view_as_complex(row2))
            return r

        arms["per_stream_plus_torch_sum"] = (ps, per_stream)
    for ch, step in arms.values():
        for _ in range(warmup):
            step()
        ch.sync()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, (ch, step) in arms.items():
            st = torch.cuda.ExternalStream(ch.cuda_stream)
            for _ in range(steps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                step()
                e1.record(st)
                ch.sync()
                times[k].append(e0.elapsed_time(e1))
    out = {"streams": S, "input_samples_per_push": L, "input_rate": sr, "output_samples_per_push": M,
           "route": "generic (k_stream_sum)" if generic else "fused (k_synth)", "arms": {}}
    if "per_stream_plus_torch_sum" not in arms and not generic:
        out["per_stream_plus_torch_sum"] = f"not run: needs about {per_stream_bytes / 2**30:.0f} GiB, {free / 2**30:.0f} GiB free"
    for k, (ch, step) in arms.items():
        ms = spread(times[k])
        b = bytes_per_push("summed" if k == "summed" else "per_stream", S, L, M)
        out["arms"][k] = {"plan": ch.plan, "ms_per_push": ms, "input_gsps": S * L / (ms["median"] * 1e-3) / 1e9,
                          "algorithmic_bytes_per_push": b, "algorithmic_gbps": b / (ms["median"] * 1e-3) / 1e9,
                          "kernel_breakdown": breakdown(ch, step)}
    for ch, _ in arms.values():
        ch.close()
    del x, row, rows
    torch.cuda.empty_cache()
    return out


def host_case(torch, rr, ctx, S, L, steps, warmup, rounds):
    sr = 48000.0
    x = torch.randn((S, L, 2), dtype=torch.float32, generator=torch.Generator().manual_seed(20264001)).pin_memory()
    su = tx_chain(rr, ctx, S)
    M = su.max_output(sr, L, 1)
    outs = [torch.empty((M, 2), dtype=torch.float32, pin_memory=True) for _ in range(2)]
    for i in range(warmup):
        su.push_summed_host_async(sr, L, 1, x.data_ptr(), L, outs[i & 1].data_ptr(), M)
    su.sync()
    per = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        for i in range(steps):
            su.push_summed_host_async(sr, L, 1, x.data_ptr(), L, outs[i & 1].data_ptr(), M)
        su.sync()
        per.append((time.perf_counter() - t0) * 1e3 / steps)
    ms = spread(per)
    out = {"streams": S, "input_samples_per_push": L, "output_samples_per_push": M,
           "timing": f"host clock around {steps} back-to-back pushes and one sync, {rounds} rounds",
           "arms": {"summed_host": {"plan": su.plan, "ms_per_push": ms, "input_gsps": S * L / (ms["median"] * 1e-3) / 1e9,
                                    "h2d_bytes_per_push": S * L * 8, "d2h_bytes_per_push": M * 8}}}
    su.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import torch

    import radiorust_b200 as rr

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device")
    ctx = rr.Context(0)
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "steps": args.steps, "warmup": args.warmup,
           "rounds": args.rounds, "cases": {}}
    for S in (1024, 4096):
        for L in (4800, 48000):
            res["cases"][f"tx_S{S}_L{L}"] = device_case(torch, rr, ctx, S, L, args.steps, args.warmup, args.rounds)
    res["cases"]["tx_host_S1024_L48000"] = host_case(torch, rr, ctx, 1024, 48000, args.steps, args.warmup, args.rounds)
    res["cases"]["generic_up3_S1024_L48000"] = device_case(torch, rr, ctx, 1024, 48000, args.steps, args.warmup, args.rounds, generic=True)
    ctx.close()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    for k, c in res["cases"].items():
        print(k, {a: (v["plan"], round(v["ms_per_push"]["median"], 3), round(v["input_gsps"], 2)) for a, v in c["arms"].items()})


if __name__ == "__main__":
    main()
