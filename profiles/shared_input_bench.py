#!/usr/bin/env python
"""Shared-input pushes against pushes of the replicated row, on the device and host-fed.

    python profiles/shared_input_bench.py --out r03_shared_input.json [--steps 20 --warmup 5]

A channelizer tunes every stream out of one wideband input.  rr_chain_push_shared[_device] reads that row once for all
streams; the replicated arm gives every stream its own copy of the row (rr_chain_push[_device]), which is what a
caller had to do before.  For every case the two arms run on two chains of the same configuration, step by step in
turn (device arms: CUDA events on each chain's stream around every push, a sync after it; host arms: a host clock
around blocks of back-to-back pushes that end in a sync).  The JSON records ms/step (median and spread),
channel-samples/s (streams x input samples per step over the step time), the kernel breakdown and plan of each arm,
the card's name and power limit, and whether the last timed step's outputs of the two arms are bit-identical.

HBM roofline fractions do not apply to the shared arm: its input is read once for all streams.
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


def lowpass(cutoff):
    def f(_bin, freq):
        return 1.0 + 0.0j if abs(freq) <= cutoff else 0.0j

    return f


def stream_shift(s: int, sr: float) -> float:
    """(577 s mod sr) - sr/2: the C3 tuning table of bench.py at 2.4 MS/s"""
    return float((s * 577) % int(sr) - sr / 2)


# name, S, input rate, chunk_len, chunks per step, output chunk, output rate, bandwidth, cutoff, expected plan
CASES = [
    ("c3_device", 4096, 2_400_000.0, 4096, 50, 2048, 48_000.0, 6_000.0, 3_000.0, "fused[filter+down]"),
    ("p200_device", 200, 9_600_000.0, 4096, 50, 2048, 48_000.0, 6_000.0, 3_000.0, None),
    ("c1_device", 512, 1_024_000.0, 4096, 50, 2048, 48_000.0, 6_000.0, 3_000.0, "front+poly[filter+down]"),
]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    line = (r.stdout.strip().splitlines() or [""])[0]
    parts = [p.strip() for p in line.split(",")]
    return {"name": parts[0] if parts else None, "power_limit": parts[1] if len(parts) > 1 else None}


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "n": len(v)}


def make_chain(rr, ctx, S, sr, n, ocl, out_rate, bw, cutoff):
    stages = [rr.FreqShifter(0.0), rr.Filter.new(lowpass(cutoff)), rr.Downsampler(ocl, out_rate, bw)]
    ch = rr.Chain(ctx, stages, "f32", n_streams=S)
    ch.set_shifts(0, [stream_shift(s, sr) for s in range(S)])
    return ch


def breakdown(ch, step, k=5):
    ch.set_timing(True)
    for _ in range(k):
        step()
    ch.sync()
    ch.kernel_time()
    b = {name: {"ms_per_step": ms / k, "launches_per_step": cnt / k} for name, (ms, cnt) in ch.kernel_breakdown().items()}
    ch.set_timing(False)
    return b


def device_case(torch, rr, ctx, case, steps, warmup):
    name, S, sr, n, chunks, ocl, out_rate, bw, cutoff, want = case
    L = n * chunks
    gen = torch.Generator(device="cuda")
    gen.manual_seed(20263000)
    row = torch.randn((L, 2), device="cuda", dtype=torch.float32, generator=gen)
    rep = row[None].expand(S, L, 2).contiguous()  # stride L (even): both arms take the TMA kernels
    sh = make_chain(rr, ctx, S, sr, n, ocl, out_rate, bw, cutoff)
    rp = make_chain(rr, ctx, S, sr, n, ocl, out_rate, bw, cutoff)
    cap = sh.max_output(sr, n, chunks) + ocl
    ysh = torch.zeros((S, cap, 2), device="cuda", dtype=torch.float32)
    yrp = torch.zeros((S, cap, 2), device="cuda", dtype=torch.float32)
    torch.cuda.synchronize()
    arms = {
        "shared": (sh, lambda: sh.push_shared_device(sr, n, chunks, row.data_ptr(), ysh.data_ptr(), cap, cap)),
        "replicated": (rp, lambda: rp.push_device(sr, n, chunks, rep.data_ptr(), L, yrp.data_ptr(), cap, cap)),
    }
    for _ in range(warmup):
        for ch, step in arms.values():
            step()
            ch.sync()
    times = {k: [] for k in arms}
    counts = {}
    for _ in range(steps):
        for k, (ch, step) in arms.items():
            st = torch.cuda.ExternalStream(ch.cuda_stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            counts[k], _ = step()
            e1.record(st)
            ch.sync()
            times[k].append(e0.elapsed_time(e1))
    # the last timed step of both arms: same pushes, same plan -> bit-identical
    plans = {k: ch.plan for k, (ch, _s) in arms.items()}
    identical = counts["shared"] == counts["replicated"] and bool(torch.equal(ysh[:, : counts["shared"]], yrp[:, : counts["replicated"]]))
    out = {"streams": S, "input_rate": sr, "chunk_len": n, "chunks_per_step": chunks, "output_rate": out_rate,
           "bit_identical_last_step": identical, "expected_plan": want, "arms": {}}
    for k, (ch, step) in arms.items():
        ms = spread(times[k])
        out["arms"][k] = {"plan": plans[k], "ms_per_step": ms, "channel_samples_per_s": S * L / (ms["median"] * 1e-3),
                          "kernel_breakdown": breakdown(ch, step)}
    sh.close()
    rp.close()
    del rep, row, ysh, yrp
    torch.cuda.empty_cache()
    return out


def host_case(torch, rr, ctx, steps, warmup, block=5):
    """C3, host-fed: rr_chain_push_shared from a pinned row against rr_chain_push of the replicated pinned input, pinned
    outputs; blocks of `block` back-to-back pushes ending in one sync, the two arms block by block in turn."""
    name, S, sr, n, chunks, ocl, out_rate, bw, cutoff, want = CASES[0]
    L = n * chunks
    row = torch.randn((L, 2), dtype=torch.float32, generator=torch.Generator().manual_seed(20263001)).pin_memory()
    rep = torch.empty((S, L, 2), dtype=torch.float32, pin_memory=True)
    for s0 in range(0, S, 256):
        rep[s0:s0 + 256] = row[None]
    sh = make_chain(rr, ctx, S, sr, n, ocl, out_rate, bw, cutoff)
    rp = make_chain(rr, ctx, S, sr, n, ocl, out_rate, bw, cutoff)
    cap = sh.max_output(sr, n, chunks) + ocl
    outs = {k: [torch.zeros((S, cap, 2), dtype=torch.float32, pin_memory=True) for _ in range(2)] for k in ("shared", "replicated")}
    cnt = {}

    def push(k, i):
        if k == "shared":
            cnt[k], _ = sh.push_shared_host_async(sr, n, chunks, row.data_ptr(), outs[k][i & 1].data_ptr(), cap, cap)
        else:
            cnt[k], _ = rp.push_host_async(sr, n, chunks, rep.data_ptr(), L, outs[k][i & 1].data_ptr(), cap, cap)

    chains = {"shared": sh, "replicated": rp}
    for k, ch in chains.items():
        for i in range(warmup):
            push(k, i)
        ch.sync()
    per_step = {k: [] for k in chains}
    blocks = max(1, (steps + block - 1) // block)
    for _ in range(blocks):
        for k, ch in chains.items():
            t0 = time.perf_counter()
            for i in range(block):
                push(k, i)
            ch.sync()
            per_step[k].append((time.perf_counter() - t0) * 1e3 / block)
    last = (block - 1) & 1  # output buffer of the last push of a block
    identical = cnt["shared"] == cnt["replicated"] and bool(torch.equal(outs["shared"][last][:, : cnt["shared"]],
                                                                         outs["replicated"][last][:, : cnt["replicated"]]))
    out = {"streams": S, "input_rate": sr, "chunk_len": n, "chunks_per_step": chunks, "output_rate": out_rate,
           "timing": f"host clock around {block} back-to-back pushes and one sync, {blocks} blocks per arm in turn",
           "bit_identical_last_step": identical, "arms": {}}
    for k, ch in chains.items():
        ms = spread(per_step[k])
        out["arms"][k] = {
            "plan": ch.plan, "ms_per_step": ms, "channel_samples_per_s": S * L / (ms["median"] * 1e-3),
            "h2d_bytes_per_step": (1 if k == "shared" else S) * L * 8, "d2h_bytes_per_step": S * cnt[k] * 8,
            "kernel_breakdown": breakdown(ch, lambda: push(k, 0)),
        }
    sh.close()
    rp.close()
    del rep, row, outs
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if args.steps < 20 or args.warmup < 5:
        raise SystemExit("at least 20 timed and 5 warm-up steps per arm")
    import torch

    import radiorust_b200 as rr

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device")
    ctx = rr.Context(0)
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0), "steps": args.steps, "warmup": args.warmup, "cases": {}}
    res["cases"]["c3_device"] = device_case(torch, rr, ctx, CASES[0], args.steps, args.warmup)
    res["cases"]["c3_host"] = host_case(torch, rr, ctx, args.steps, args.warmup)
    for case in CASES[1:]:
        res["cases"][case[0]] = device_case(torch, rr, ctx, case, args.steps, args.warmup)
    ctx.close()
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    for k, c in res["cases"].items():
        a, b = c["arms"]["shared"], c["arms"]["replicated"]
        print(f"{k}: shared {a['ms_per_step']['median']:.3f} ms ({a['plan']}), replicated {b['ms_per_step']['median']:.3f} ms "
              f"({b['plan']}), identical {c['bit_identical_last_step']}")


if __name__ == "__main__":
    main()
