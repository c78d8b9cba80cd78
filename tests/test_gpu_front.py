"""GPU parity tests of the rank-reduced path (k_front + k_poly2, DESIGN.md 4.1) through the C ABI.

The path is chosen automatically for complex-f32 FreqShifter/Filter -> Downsampler chains with integer
decimation P, P = 2 (mod 4), whose fused filter factors to rank <= 10.  Everything here is compared
with the numpy oracle (relative L2 <= 1e-5) and with the library's own other paths.
"""
import os

import numpy as np
import pytest

from oracle import radiorust_oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-5


@pytest.fixture(scope="module")
def ctx():
    import radiorust_b200 as rr

    c = rr.Context(0)
    yield c
    c.close()


def oracle_chain(shift, cutoff, ocl, out_rate, bw, sr, x, n, with_nco=True):
    blocks = ([orc.FreqShifter("f32", 1.0, shift)] if with_nco else []) + [
        orc.Filter.new("f32", orc.lowpass(cutoff)), orc.Downsampler("f32", ocl, out_rate, bw)]
    return orc.Chain(blocks).run(sr, x, n)


def gpu_chain(ctx, shifts, cutoff, ocl, out_rate, bw, sr, x, n, pushes, with_nco=True, env=None):
    import radiorust_b200 as rr

    old = {}
    for k, v in (env or {}).items():
        old[k] = os.environ.get(k)
        os.environ[k] = v
    try:
        stages = ([rr.FreqShifter(0.0)] if with_nco else []) + [rr.Filter.new(orc.lowpass(cutoff)), rr.Downsampler(ocl, out_rate, bw)]
        ch = rr.Chain(ctx, stages, "f32", n_streams=x.shape[0])
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    if with_nco:
        ch.set_shifts(0, list(shifts))
    got, plans, pos = [], [], 0
    for k in pushes:
        y, rate = ch.push(sr, np.ascontiguousarray(x[:, pos * n:(pos + k) * n]), n)
        if y.shape[1]:
            assert rate == out_rate
        got.append(y.copy())
        plans.append(ch.plan)
        pos += k
    ch.close()
    return np.concatenate(got, axis=1), plans


@pytest.mark.parametrize("sr,n,cutoff,out_rate,bw,ocl,P", [
    (2_400_000.0, 4096, 3000.0, 48000.0, 6000.0, 2048, 50),   # C3, the benchmarked configuration
    (1_440_000.0, 4096, 3000.0, 48000.0, 6000.0, 100, 30),
    (480_000.0, 1024, 8000.0, 48000.0, 20000.0, 17, 10),      # odd output chunking
    (3_360_000.0, 4096, 3000.0, 48000.0, 6000.0, 256, 70),
    (960_000.0, 2048, 10000.0, 48000.0, 20000.0, 17, 20),     # P = 0 (mod 4): padded tile pitch
    (3_072_000.0, 4096, 3000.0, 48000.0, 6000.0, 64, 64),
    (4_800_000.0, 4096, 3000.0, 48000.0, 6000.0, 1024, 100),
])
def test_front_path_rates(ctx, sr, n, cutoff, out_rate, bw, ocl, P):
    S = 3
    pushes = [3, 1, 9, 2, 11, 1, 14]
    total = sum(pushes)
    x = np.stack([orc.synth_noise(5100 + 7 * s + P, total * n, "f32") for s in range(S)])
    shifts = [sr / 7.0, -sr / 3.0 + 11.0, 0.0]
    got, plans = gpu_chain(ctx, shifts, cutoff, ocl, out_rate, bw, sr, x, n, pushes)
    assert any("front+poly2" in p for p in plans), plans
    for s in range(S):
        want = oracle_chain(shifts[s], cutoff, ocl, out_rate, bw, sr, x[s], n)
        assert want.shape == got[s].shape
        assert orc.rel_l2(got[s], want) <= TOL


def test_front_equals_other_paths(ctx):
    """k_front + k_poly2 vs k_poly2 on all branches vs k_poly vs the stateful overlap-save kernels."""
    sr, n, S = 2_400_000.0, 4096, 2
    pushes = [4, 20, 6]
    x = np.stack([orc.synth_noise(777 + s, sum(pushes) * n, "f32") for s in range(S)])
    shifts = [-577000.0, 1_000_001.0]
    args = (shifts, 3000.0, 64, 48000.0, 6000.0, sr, x, n, pushes)
    a, pa = gpu_chain(ctx, *args)
    b, pb = gpu_chain(ctx, *args, env={"RR_DISABLE_FRONT": "1"})
    c, pc = gpu_chain(ctx, *args, env={"RR_DISABLE_POLY2": "1"})
    d, pd = gpu_chain(ctx, *args, env={"RR_DISABLE_POLY": "1"})
    assert any("front+poly2" in p for p in pa)
    assert any("poly2[" in p for p in pb) and not any("front" in p for p in pb)
    assert any("poly[" in p for p in pc) and not any("poly2" in p for p in pc)
    assert not any("poly" in p for p in pd)
    for other in (b, c, d):
        assert other.shape == a.shape
        assert orc.rel_l2(a, other) < 3e-6


def test_front_without_nco_and_single_chunk_pushes(ctx):
    """Filter -> Downsampler without a FreqShifter; pushes of one chunk never hold a whole transform window,
    so every block takes the thread-local edge loads and the history comes from hist2."""
    sr, n, S = 2_400_000.0, 4096, 5
    pushes = [1] * 9 + [8] + [1] * 3
    x = np.stack([orc.synth_noise(31 + s, sum(pushes) * n, "f32") for s in range(S)])
    got, plans = gpu_chain(ctx, None, 3000.0, 128, 48000.0, 6000.0, sr, x, n, pushes, with_nco=False)
    assert any("front+poly2" in p for p in plans), plans
    for s in range(S):
        want = oracle_chain(0.0, 3000.0, 128, 48000.0, 6000.0, sr, x[s], n, with_nco=False)
        assert orc.rel_l2(got[s], want) <= TOL


def test_front_events_retune_and_redesign(ctx):
    import radiorust_b200 as rr

    sr, n = 2_400_000.0, 4096
    x = orc.synth_noise(99, 60 * n, "f32")
    stages = [rr.FreqShifter(250000.0), rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(96, 48000.0, 6000.0)]
    ch = rr.Chain(ctx, stages, "f32")
    ob = [orc.FreqShifter("f32", 1.0, 250000.0), orc.Filter.new("f32", orc.lowpass(3000.0)), orc.Downsampler("f32", 96, 48000.0, 6000.0)]
    oc = orc.Chain(ob)
    got, want, plans = [], [], []

    def feed(lo, hi):
        y, _ = ch.push(sr, x[lo * n:hi * n], n)
        plans.append(ch.plan)
        got.append(y[0].copy())
        for k in range(lo, hi):
            for m in oc.push(orc.Samples(sr, x[k * n:(k + 1) * n])):
                if isinstance(m, orc.Samples):
                    want.append(m.chunk)

    feed(0, 12)
    feed(12, 20)
    ch.event(True)                       # interrupt: the Filter drops its history (filters.rs:262-267)
    oc.push(orc.DISCONNECTION)
    feed(20, 30)
    ch.set_shift(0, -123456.0)           # phase-continuous retune (transform.rs:322-327)
    ob[0].set_shift(-123456.0)
    feed(30, 40)
    ch.update_filter(1, orc.lowpass(4500.0))   # redesign: new rank tables, history dropped
    ob[1].update(orc.lowpass(4500.0))
    feed(40, 52)
    ch.set_fast_path(False)              # the stateful kernels take over from hist2
    feed(52, 56)
    ch.set_fast_path(True)
    feed(56, 60)
    ch.close()
    assert sum("front+poly2" in p for p in plans) >= 4, plans
    g, w = np.concatenate(got), np.concatenate(want)
    assert g.shape == w.shape
    assert orc.rel_l2(g, w) <= TOL


def test_front_full_chunk_structure_properties(ctx):
    """BASELINE-sized pushes (50 chunks of 4096 per stream per push) on a reduced number of streams, through
    properties that need no oracle run at that size: streams are independent and deterministic (identical
    inputs give bit-identical outputs wherever they sit in the batch), and the chain is linear."""
    sr, n, S, chunks = 2_400_000.0, 4096, 24, 100
    base = orc.synth_noise(4242, chunks * n, "f32")
    other = orc.synth_noise(4243, chunks * n, "f32")
    x = np.stack([base if s % 3 == 0 else (other if s % 3 == 1 else (0.5 * base - 2.0 * other).astype(np.complex64)) for s in range(S)])
    shifts = [123457.0] * S
    got, plans = gpu_chain(ctx, shifts, 3000.0, 2048, 48000.0, 6000.0, sr, x, n, [50, 50])
    assert all("front+poly2" in p for p in plans), plans
    for s in range(3, S):
        assert np.array_equal(got[s], got[s % 3]), s          # independence + determinism
    lin = 0.5 * got[0] - 2.0 * got[1]
    assert orc.rel_l2(got[2], lin) < 5e-6                      # linearity
    want = oracle_chain(123457.0, 3000.0, 2048, 48000.0, 6000.0, sr, x[0], n)
    assert orc.rel_l2(got[0], want) <= TOL


def test_front_runs_are_bit_reproducible(ctx):
    """Two fresh chains on the same input give bit-identical outputs (no atomics in the arithmetic, no
    order-dependent reductions): a cheap detector of shared-memory races in the warp-autonomous kernels.
    An odd number of streams leaves one CTA half of k_poly2 idle; 37 streams walk several persistent halves."""
    sr, n, S = 2_400_000.0, 4096, 37
    pushes = [26, 3, 31]
    x = np.stack([orc.synth_noise(9000 + s, sum(pushes) * n, "f32") for s in range(S)])
    shifts = [float((s * 577) % 2_400_000 - 1_200_000) for s in range(S)]   # SURVEY.md 8(d), config C3
    args = (shifts, 3000.0, 2048, 48000.0, 6000.0, sr, x, n, pushes)
    a, pa = gpu_chain(ctx, *args)
    for _ in range(3):
        b, _ = gpu_chain(ctx, *args)
        assert np.array_equal(a, b)
    assert any("front+poly2" in p for p in pa)
    for s in (0, 17, 36):
        want = oracle_chain(shifts[s], 3000.0, 2048, 48000.0, 6000.0, sr, x[s], n)
        assert orc.rel_l2(a[s], want) <= TOL


def test_front_full_baseline_size_on_device(ctx):
    """BASELINE.json config C3 at its full single-GPU size -- 4096 streams x 50 chunks x 4096 samples per push,
    device resident (6.7 GB of input), three pushes of the same samples -- with every stream checked.  The chain is
    linear for a fixed shift: stream s is a_s*A + b_s*B (seeded weights of order 1) with shift class s mod 7 (7 is
    coprime to the SM count, so the stream a persistent CTA runs just before s has another shift and other weights),
    and must come out as a_s*ref(A, k) + b_s*ref(B, k) with the f64 oracle's ref: per stream, rel-L2 <= 3e-6 and
    max |err| / rms <= 3e-5 (tests/test_gpu_layout.py explains the bounds)."""
    import math

    import torch

    import radiorust_b200 as rr

    sr, n, S, C, K = 2_400_000.0, 4096, 4096, 50, 7
    length = C * n
    assert math.gcd(torch.cuda.get_device_properties(0).multi_processor_count, K) == 1
    A = orc.synth_noise(20260000 + 3 * 100000, length, "f64")
    B = orc.synth_noise(20260000 + 3 * 100000 + 1, length, "f64")
    rng = np.random.default_rng(20260000 + 3 * 100000 + 2)
    wa, wb = (0.5 + rng.random((2, S))) * np.exp(2j * np.pi * rng.random((2, S)))
    A_d, B_d, a_d, b_d = (torch.from_numpy(v).cuda() for v in (A, B, wa, wb))
    x = torch.empty((S, length), device="cuda", dtype=torch.complex64)
    for s0 in range(0, S, 128):
        x[s0:s0 + 128] = (a_d[s0:s0 + 128, None] * A_d[None] + b_d[s0:s0 + 128, None] * B_d[None]).to(torch.complex64)
    del A_d, B_d
    class_shift = [float((k * 577 * 293) % 2_400_000 - 1_200_000) for k in range(K)]   # SURVEY.md 8(d) style
    chain = rr.Chain(ctx, [rr.FreqShifter(0.0), rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(2048, 48000.0, 6000.0)],
                     "f32", n_streams=S)
    chain.set_shifts(0, [class_shift[s % K] for s in range(S)])
    cap = chain.max_output(sr, n, C + 1) + 2048
    y = torch.zeros((S, cap), device="cuda", dtype=torch.complex64)
    torch.cuda.synchronize()
    outs = []
    for push in range(3):
        cnt, rate = chain.push_device(sr, n, C, x.data_ptr(), length, y.data_ptr(), cap, cap)
        chain.sync()
        torch.cuda.synchronize()
        assert rate == 48000.0 and cnt > 0 and cnt % 2048 == 0
        # push 0: start-up chunks + k_front + k_poly2; push 1 (steady state): k_fused
        assert ("front+poly2" if push == 0 else "fused[") in chain.plan, chain.plan
        outs.append(y[:, :cnt].cpu().numpy())
    chain.close()
    del x, y
    torch.cuda.empty_cache()
    got = np.concatenate(outs, axis=1)
    ref = []
    for base in (A, B):
        ref.append(np.stack([orc.Chain([orc.FreqShifter("f64", 1.0, class_shift[k]), orc.Filter.new("f64", orc.lowpass(3000.0)),
                                        orc.Downsampler("f64", 2048, 48000.0, 6000.0)]).run(sr, np.concatenate([base, base, base]), n)
                             for k in range(K)]))
    assert got.shape == (S, ref[0].shape[1]), (got.shape, ref[0].shape)
    M = got.shape[1]
    for s0 in range(0, S, 512):
        cls = np.arange(s0, s0 + 512) % K
        want = wa[s0:s0 + 512, None] * ref[0][cls] + wb[s0:s0 + 512, None] * ref[1][cls]
        err = got[s0:s0 + 512].astype(np.complex128) - want
        den = np.linalg.norm(want, axis=1)
        rel = np.linalg.norm(err, axis=1) / den
        mx = np.abs(err).max(axis=1) / (den / math.sqrt(M))
        bad = np.flatnonzero(~((rel <= 3e-6) & (mx <= 3e-5)))
        assert bad.size == 0, (s0 + bad[:8], rel[bad[:8]], mx[bad[:8]])


def test_chain_destroy_releases_device_memory(ctx):
    """Creating and destroying chains (incl. the front end's scratch buffers) must not leak device memory."""
    import torch

    import radiorust_b200 as rr

    sr, n, S = 2_400_000.0, 4096, 64
    x = np.stack([orc.synth_noise(3 + s, 20 * n, "f32") for s in range(S)])

    def once():
        ch = rr.Chain(ctx, [rr.FreqShifter(1000.0), rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(64, 48000.0, 6000.0)], "f32", n_streams=S)
        ch.push(sr, x, n)
        assert "front+poly2" in ch.plan
        ch.close()

    once()
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for _ in range(5):
        once()
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 < 8 * 1024 * 1024, (free0, free1)


def test_kept_u_rows_match_recomputed_history(ctx, monkeypatch):
    """Pushes that follow a front-end push reuse its last Lmax rows of u instead of recomputing them from hist2
    (`k_front` copies them over); RR_DISABLE_UCACHE=1 recomputes.  Both match the oracle, through
    ragged push sizes, a retune (the kept rows stay valid: the mixed signal is phase continuous), an interrupt and a
    filter update (both start a new segment: nothing is kept across them)."""
    import radiorust_b200 as rr

    sr, n, S = 2_400_000.0, 4096, 3
    lp = orc.lowpass(3000.0)
    rng = np.random.default_rng(99)
    script = [3, 1, 1, 2, 1, "retune", 1, 5, 1, "interrupt", 1, 1, 1, 2, "update", 1, 1, 1, 1]
    total = sum(k for k in script if isinstance(k, int))
    x = (rng.standard_normal((S, total * n)) + 1j * rng.standard_normal((S, total * n))).astype(np.complex64)

    def run(disable):
        if disable:
            monkeypatch.setenv("RR_DISABLE_UCACHE", "1")
        else:
            monkeypatch.delenv("RR_DISABLE_UCACHE", raising=False)
        ch = rr.Chain(ctx, [rr.FreqShifter(12345.0), rr.Filter.new(lp), rr.Downsampler(16, 48000.0, 6000.0)], "f32", n_streams=S)
        ch.set_timing(True)
        outs, pos = [], 0
        for k in script:
            if k == "retune":
                ch.set_shift(0, -77777.0)
            elif k == "interrupt":
                ch.event(True)
            elif k == "update":
                ch.update_filter(1, orc.lowpass(2500.0))
            else:
                y, _ = ch.push(sr, x[:, pos * n:(pos + k) * n], n)
                outs.append(y.copy())
                pos += k
        ch.kernel_time()
        bd = ch.kernel_breakdown()
        ch.close()
        return np.concatenate(outs, axis=1), bd

    got, bd = run(False)
    got_nc, bd_nc = run(True)
    assert bd["k_front"][1] == bd_nc["k_front"][1] >= 8
    for s in range(S):
        blocks = [orc.FreqShifter("f32", 1.0, 12345.0), orc.Filter.new("f32", lp), orc.Downsampler("f32", 16, 48000.0, 6000.0)]
        chain = orc.Chain(blocks)
        want, pos = [], 0
        for k in script:
            if k == "retune":
                blocks[0].set_shift(-77777.0)
            elif k == "interrupt":
                chain.push(orc.Event("x", True))
            elif k == "update":
                blocks[1].update(orc.lowpass(2500.0))
            else:
                for c in range(k):
                    want += [m.chunk for m in chain.push(orc.Samples(sr, x[s, (pos + c) * n:(pos + c + 1) * n])) if isinstance(m, orc.Samples)]
                pos += k
        want = np.concatenate(want)
        assert got.shape[1] == len(want) == got_nc.shape[1]
        assert orc.rel_l2(got[s], want) <= 1e-5 and orc.rel_l2(got_nc[s], want) <= 1e-5
        assert orc.rel_l2(got[s], got_nc[s]) <= 2e-6


def test_short_pushes_of_many_streams_group_streams_per_inverse_round(ctx, monkeypatch):
    """More streams than CTA halves and at most three low-rate blocks per stream (pushes of 1-15 chunks): k_poly2 takes
    runs of streams as the blocks of one launch "stream" (PolyArgs::sab_*).  Same arithmetic per block, so the result is
    bit-identical to RR_DISABLE_SAB=1; 601 streams leave two padded, non-existent streams in the last run."""
    import radiorust_b200 as rr

    sr, n, S = 2_400_000.0, 4096, 601
    lp = orc.lowpass(3000.0)
    rng = np.random.default_rng(7)
    sizes = [3, 1, 2, 1, 5, 1, 1, 9, 2, 12, 7, 16, 1]  # one, two and three low-rate blocks per stream; 16 chunks: four (per-stream form)
    total = sum(sizes)
    x = (rng.standard_normal((S, total * n)) + 1j * rng.standard_normal((S, total * n))).astype(np.complex64)
    shifts = [(s * 577) % 2_400_000 - 1_200_000 for s in range(S)]

    def run(disable):
        if disable:
            monkeypatch.setenv("RR_DISABLE_SAB", "1")
        else:
            monkeypatch.delenv("RR_DISABLE_SAB", raising=False)
        ch = rr.Chain(ctx, [rr.FreqShifter(0.0), rr.Filter.new(lp), rr.Downsampler(16, 48000.0, 6000.0)], "f32", n_streams=S)
        ch.set_shifts(0, shifts)
        outs, pos = [], 0
        for k in sizes:
            y, _ = ch.push(sr, x[:, pos * n:(pos + k) * n], n)
            outs.append(y.copy())
            pos += k
        ch.close()
        return np.concatenate(outs, axis=1)

    got, ref = run(False), run(True)
    assert got.shape == ref.shape and got.shape[1] > 1000
    assert np.array_equal(got, ref)
    for s in (0, 299, 600):
        chain = orc.Chain([orc.FreqShifter("f32", 1.0, float(shifts[s])), orc.Filter.new("f32", lp), orc.Downsampler("f32", 16, 48000.0, 6000.0)])
        want = chain.run(sr, x[s], n)
        assert len(want) == got.shape[1] and orc.rel_l2(got[s], want) <= 1e-5
