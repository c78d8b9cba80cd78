"""Shared-input pushes: every stream of a chain reads one input row (rr_chain_push_shared[_device]).

A channelizer tunes all its streams out of one wideband input.  The shared row is pushed from a device buffer with NaN
on both sides, so a kernel that reads outside [0, len) -- or a TMA copy that still addresses row s of a one-row map --
fails.  Two checks apply to every push:

- twin: a second chain with the same configuration gets the row replicated into every stream through
  rr_chain_push_device (rows at an even stride, so that both take the same plan).  Plans must match, and every stream
  must be bit-identical to the twin's.
- oracle: stream s has shift class s mod 7 (coprime to the SM count: the stream a persistent CTA handles just before s
  has another shift) and is checked against the f64 oracle of its class with test_gpu_layout.BOUNDS, per stream.

Worst per-stream values measured on a B200 are in DESIGN.md 4.8.
"""
import math

import numpy as np
import pytest

from oracle import radiorust_oracle as orc
from test_gpu_layout import BOUNDS, FAMILIES, K, Cfg, class_shifts, down_chain, family, oracle_run

pytestmark = pytest.mark.gpu

TMA_OFF_LEAD = 3  # f32 samples in front of the row: 24 bytes, off 16-byte alignment


@pytest.fixture(scope="module")
def ctx():
    import radiorust_b200 as rr

    c = rr.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sm():
    import torch

    n = torch.cuda.get_device_properties(0).multi_processor_count
    assert math.gcd(n, K) == 1, n
    return n


def clear_env(monkeypatch):
    for v in ("RR_FUSED_MIN_STREAMS", "RR_DISABLE_FUSED", "RR_DISABLE_FRONT", "RR_DISABLE_POLY", "RR_DISABLE_POLY2"):
        monkeypatch.delenv(v, raising=False)


def make_chain(ctx, cfg, S, shifts):
    import radiorust_b200 as rr

    ch = rr.Chain(ctx, cfg.gpu(), cfg.flt, n_streams=S)
    if cfg.nco is not None:
        ch.set_shifts(cfg.nco, [shifts[s % K] for s in range(S)])
    if not cfg.fast_path:
        ch.set_fast_path(False)
    return ch


def cdtype(flt):
    import torch

    return (torch.complex64, 8) if flt == "f32" else (torch.complex128, 16)


def aligned_lead(flt):
    return 2 if flt == "f32" else 1  # 16 bytes


def shared_row(x, flt, lead):
    """x (host, f64) as one device row `lead` samples into a buffer with NaN on both sides; returns (buffer, ptr)."""
    import torch

    cdt, esz = cdtype(flt)
    buf = torch.full((lead + len(x) + 5,), float("nan"), dtype=cdt, device="cuda")
    buf[lead:lead + len(x)] = torch.from_numpy(x).to(cdt).cuda()
    return buf, buf.data_ptr() + lead * esz


def replicated_rows(x, S, flt, lead):
    """x in every one of S rows at an even stride (NaN padding); returns (buffer, ptr, stride)."""
    import torch

    cdt, esz = cdtype(flt)
    L = len(x)
    stride = L + 3 + (L + 3) % 2
    buf = torch.full((lead + S * stride,), float("nan"), dtype=cdt, device="cuda")
    v = buf.as_strided((S, L), (stride, 1), lead)
    v[:] = torch.from_numpy(x).to(cdt).cuda()[None, :]
    return buf, v.data_ptr(), stride


class Pair:
    """A chain fed shared pushes and its twin fed the replicated row through rr_chain_push_device."""

    def __init__(self, ctx, cfg, S, shifts):
        self.cfg, self.S = cfg, S
        self.a = make_chain(ctx, cfg, S, shifts)
        self.b = make_chain(ctx, cfg, S, shifts)

    def close(self):
        self.a.close()
        self.b.close()

    def push(self, x, lead, shared=True):
        """One push of row x to both; asserts the same plan and bit-identical outputs.  shared=False feeds the
        first chain the replicated row too (per-stream push).  Returns ([S, M] output, plan)."""
        import torch

        cfg, S, n = self.cfg, self.S, self.cfg.n
        k = len(x) // n
        cdt, _ = cdtype(cfg.flt)
        cap = self.a.max_output(cfg.sr, n, k)
        assert cap == self.b.max_output(cfg.sr, n, k)
        ostride = cap + 1
        ya = torch.full((max(S * ostride, 1),), float("nan"), dtype=cdt, device="cuda")
        yb = torch.full((max(S * ostride, 1),), float("nan"), dtype=cdt, device="cuda")
        rep, rptr, rstride = replicated_rows(x, S, cfg.flt, lead)
        if shared:
            row, ptr = shared_row(x, cfg.flt, lead)
        torch.cuda.synchronize()
        if shared:
            ca, _ = self.a.push_shared_device(cfg.sr, n, k, ptr, ya.data_ptr(), cap, ostride)
        else:
            ca, _ = self.a.push_device(cfg.sr, n, k, rptr, rstride, ya.data_ptr(), cap, ostride)
        cb, _ = self.b.push_device(cfg.sr, n, k, rptr, rstride, yb.data_ptr(), cap, ostride)
        self.a.sync()
        self.b.sync()
        assert ca == cb
        assert self.a.plan == self.b.plan, (self.a.plan, self.b.plan)
        ga = ya.as_strided((S, ca), (ostride, 1)).cpu().numpy()
        gb = yb.as_strided((S, cb), (ostride, 1)).cpu().numpy()
        assert np.array_equal(ga, gb), f"shared push differs from the replicated twin ({self.a.plan})"
        return ga, self.a.plan


def references(cfg, x, shifts):
    """[K, M] f64 oracle output of row x per shift class (one row when the chain has no FreqShifter)."""
    return np.stack([oracle_run(cfg.oracle(shifts[k] if cfg.nco is not None else 0.0), cfg.sr, x, cfg.n)
                     for k in range(K if cfg.nco is not None else 1)])


def check_streams(got, ref, flt, label, streams=None):
    """Stream s (streams[i] for row i of got) against ref[s mod classes]; returns (worst rel, worst max)."""
    S, M = got.shape
    assert M == ref.shape[1] and M > 0, (got.shape, ref.shape)
    streams = np.arange(S) if streams is None else np.asarray(streams)
    lim_rel, lim_max = BOUNDS[flt]
    rel = np.empty(S)
    mx = np.empty(S)
    for s0 in range(0, S, 4096):
        s1 = min(S, s0 + 4096)
        want = ref[streams[s0:s1] % ref.shape[0]]
        err = got[s0:s1].astype(np.complex128) - want
        den = np.linalg.norm(want, axis=1)
        rel[s0:s1] = np.linalg.norm(err, axis=1) / den
        mx[s0:s1] = np.abs(err).max(axis=1) / (den / math.sqrt(M))
    bad = np.flatnonzero(~((rel <= lim_rel) & (mx <= lim_max)))
    wr, wm = float(np.nanmax(rel)), float(np.nanmax(mx))
    print(f"\nSHARED {label}: {flt} streams={S} outputs={M} worst rel {wr:.2e} max {wm:.2e}")
    assert bad.size == 0, (label, f"{bad.size} of {S} streams out of bounds, first {streams[bad[:8]].tolist()}",
                           rel[bad[:8]].tolist(), mx[bad[:8]].tolist())
    return wr, wm


def run_pushes(pair, x, lead):
    """cfg.pushes consecutive windows of x through the pair; returns ([S, M] outputs, plans)."""
    outs, plans, pos = [], [], 0
    for k in pair.cfg.pushes:
        L = k * pair.cfg.n
        got, plan = pair.push(x[pos:pos + L], lead)
        outs.append(got)
        plans.append(plan)
        pos += L
    return np.concatenate(outs, axis=1), plans


# ---- chains whose first stage is not a Filter ------------------------------------------------------------------------
def first_stage_family(name):
    import radiorust_b200 as rr

    if name == "fmdemod_first":   # FmDemod reads the shared row; a per-stream shift behind it (f64: exact angles)
        return Cfg("f64", 240_000.0, 1024, [2, 3, 1],
                   lambda: [rr.FmDemod(75000.0), rr.FreqShifter(0.0), rr.Filter.new(orc.lowpass(15000.0)), rr.Downsampler(256, 48000.0, 15000.0)],
                   lambda shift: [orc.FmDemod("f64", 75000.0), orc.FreqShifter("f64", 1.0, shift), orc.Filter.new("f64", orc.lowpass(15000.0)),
                                  orc.Downsampler("f64", 256, 48000.0, 15000.0)], nco=1, plan="fmdemod")
    if name == "fourier_pow2":    # f64 here and below: the bounds of an f32 transform sit at those of the f64 oracle
        return Cfg("f64", 48000.0, 1024, [1, 3, 2], lambda: [rr.Fourier(), rr.GainControl(0.5)],
                   lambda _s: [orc.Fourier("f64"), orc.GainControl("f64", 0.5)], nco=None, plan="fourier")
    if name == "fourier_direct":  # a length outside the FFT plans: the direct DFT
        return Cfg("f64", 48000.0, 1000, [1, 3, 2], lambda: [rr.Fourier(center_dc=True)],
                   lambda _s: [orc.Fourier("f64", center_dc=True)], nco=None, plan="fourier")
    if name == "fmmod":           # the phase accumulator in f64: the device follows the reference's rounding exactly
        return Cfg("f64", 48000.0, 512, [1, 3, 2], lambda: [rr.FmMod(5000.0), rr.FreqShifter(0.0)],
                   lambda shift: [orc.FmMod("f64", 5000.0), orc.FreqShifter("f64", 1.0, shift)], nco=1, plan="fmmod")
    if name == "gain_first":      # GainControl reads the row, then the C3 path with the NCO in a stand-alone kernel
        return Cfg("f32", 2_400_000.0, 4096, [3, 5, 2], lambda: [rr.GainControl(2.0), rr.FreqShifter(0.0), rr.Filter.new(orc.lowpass(3000.0)),
                                                                rr.Downsampler(64, 48000.0, 6000.0)],
                   lambda shift: [orc.GainControl("f64", 2.0), orc.FreqShifter("f64", 1.0, shift), orc.Filter.new("f64", orc.lowpass(3000.0)),
                                  orc.Downsampler("f64", 64, 48000.0, 6000.0)], nco=1, plan="gain")
    raise KeyError(name)


FIRST_STAGE = ["fmdemod_first", "fourier_pow2", "fourier_direct", "fmmod", "gain_first"]


def row_signal(cfg, total, seed):
    if cfg.plan == "fmdemod":
        return orc.synth_fm_station(seed, total, cfg.sr).astype(np.complex128)
    return orc.synth_noise(seed, total, "f64")


# ---- 1. family sweep -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", FAMILIES + FIRST_STAGE)
def test_family_sweep(ctx, sm, monkeypatch, name):
    """Every path family of test_gpu_layout plus chains that start with another stage, fed one shared row.  The k_fused
    families run with the threshold forced to one stream and S = SM + 1 (one CTA takes two streams)."""
    clear_env(monkeypatch)
    cfg = family(name) if name in FAMILIES else first_stage_family(name)
    fused = name.startswith("fused_p")
    if fused:
        monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    S = sm + 1 if fused else 2 * K + 3
    x = row_signal(cfg, sum(cfg.pushes) * cfg.n, 7100 + (FAMILIES + FIRST_STAGE).index(name))
    shifts = class_shifts(cfg.sr)
    ref = references(cfg, x, shifts)
    pair = Pair(ctx, cfg, S, shifts)
    try:
        got, plans = run_pushes(pair, x, aligned_lead(cfg.flt))
    finally:
        pair.close()
    print(f"\nPLANS shared {name}: {plans}")
    assert any(cfg.plan in p for p in plans), plans
    check_streams(got, ref, cfg.flt, name)


# ---- 2. misaligned row -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["fused_p50", "front_poly2", "front16_poly", "rechunk_view"])
def test_misaligned_row(ctx, sm, monkeypatch, name):
    """A row one f32 sample off 16 bytes turns TMA off: the non-TMA plan runs, bit-identical to a twin whose rows have
    the same misalignment, and correct."""
    clear_env(monkeypatch)
    cfg = family(name)
    if name.startswith("fused_p"):
        monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    S = sm + 1
    x = orc.synth_noise(7200 + len(name), sum(cfg.pushes) * cfg.n, "f64")
    shifts = class_shifts(cfg.sr)
    ref = references(cfg, x, shifts)
    pair = Pair(ctx, cfg, S, shifts)
    try:
        got, plans = run_pushes(pair, x, TMA_OFF_LEAD)
    finally:
        pair.close()
    print(f"\nPLANS shared misaligned {name}: {plans}")
    assert any(cfg.tma_plan in p for p in plans), plans
    assert not any(bad in p for p in plans for bad in cfg.not_tma), plans
    check_streams(got, ref, cfg.flt, f"misaligned/{name}")


# ---- 3. host path ---------------------------------------------------------------------------------------------------------
def test_host_push_equals_device_push(ctx, sm, monkeypatch):
    """push_shared (host row) equals push_shared_device bit for bit, with the fused path in steady state; then three
    back-to-back push_shared_host_async calls from pinned buffers with a single sync."""
    import torch

    clear_env(monkeypatch)
    monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    cfg = family("fused_p50")
    S = sm + 1
    n = cfg.n
    pushes = [3, 5, 2, 4, 1, 3]
    x = orc.synth_noise(7300, sum(pushes) * n, "f64")
    x32 = x.astype(np.complex64)
    shifts = class_shifts(cfg.sr)
    host = make_chain(ctx, cfg, S, shifts)
    dev = make_chain(ctx, cfg, S, shifts)
    try:
        pos, outs = 0, []
        for i, k in enumerate(pushes[:3]):
            L = k * n
            yh, _ = host.push_shared(cfg.sr, x32[pos:pos + L], n)
            cap = dev.max_output(cfg.sr, n, k)
            row, ptr = shared_row(x[pos:pos + L], "f32", 2)
            yd = torch.empty((S, max(cap, 1)), dtype=torch.complex64, device="cuda")
            torch.cuda.synchronize()
            cnt, _ = dev.push_shared_device(cfg.sr, n, k, ptr, yd.data_ptr(), cap, yd.shape[1])
            dev.sync()
            assert host.plan == dev.plan, (host.plan, dev.plan)
            assert yh.shape[1] == cnt and np.array_equal(yh, yd[:, :cnt].cpu().numpy()), i
            outs.append(yh.copy())
            pos += L
        assert "fused[" in host.plan, host.plan
        # three asynchronous host pushes, one sync
        ins, youts, counts = [], [], []
        for k in pushes[3:]:
            L = k * n
            pin = ctx.pinned_array((L,), np.complex64)
            pin[:] = x32[pos:pos + L]
            cap = host.max_output(cfg.sr, n, k)
            pout = ctx.pinned_array((S, max(cap, 1)), np.complex64)
            pout[:] = np.nan
            cnt, _ = host.push_shared_host_async(cfg.sr, n, k, pin.ctypes.data, pout.ctypes.data, cap, pout.shape[1])
            ins.append(pin)
            youts.append(pout)
            counts.append(cnt)
            pos += L
        host.sync()
        pos = sum(pushes[:3]) * n
        for k, pout, cnt in zip(pushes[3:], youts, counts):
            L = k * n
            cap = dev.max_output(cfg.sr, n, k)
            row, ptr = shared_row(x[pos:pos + L], "f32", 2)
            yd = torch.empty((S, max(cap, 1)), dtype=torch.complex64, device="cuda")
            torch.cuda.synchronize()
            c2, _ = dev.push_shared_device(cfg.sr, n, k, ptr, yd.data_ptr(), cap, yd.shape[1])
            dev.sync()
            assert c2 == cnt and np.array_equal(np.asarray(pout)[:, :cnt], yd[:, :cnt].cpu().numpy())
            outs.append(np.array(pout[:, :cnt]))
            pos += L
    finally:
        host.close()
        dev.close()
    ref = references(Cfg(cfg.flt, cfg.sr, n, pushes, cfg.gpu, cfg.oracle), x, shifts)
    check_streams(np.concatenate(outs, axis=1), ref, "f32", "host")


# ---- 4. mixed pushes and state changes -----------------------------------------------------------------------------------
def test_mixed_and_stateful(ctx, sm, monkeypatch):
    """On one chain: shared pushes, per-stream pushes of the replicated row, an interrupt event, a retune of every
    stream and a filter update in between.  The twin sees only replicated pushes; bit-identical at every step."""
    clear_env(monkeypatch)
    monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    cfg = family("fused_p50")
    S = sm + 1
    n = cfg.n
    x = orc.synth_noise(7400, 40 * n, "f64")
    shifts = class_shifts(cfg.sr)
    pair = Pair(ctx, cfg, S, shifts)
    retune = [-shifts[(s + 3) % K] / 2 for s in range(S)]
    steps = [("shared", 3), ("shared", 4), ("per_stream", 2), ("shared", 5), ("event", 0), ("shared", 3), ("shared", 2),
             ("retune", 0), ("shared", 4), ("per_stream", 3), ("filter", 0), ("shared", 3), ("shared", 4), ("per_stream", 1),
             ("shared", 1)]
    plans, pos = [], 0
    try:
        for what, k in steps:
            if what == "event":
                pair.a.event(True)
                pair.b.event(True)
            elif what == "retune":
                pair.a.set_shifts(cfg.nco, retune)
                pair.b.set_shifts(cfg.nco, retune)
            elif what == "filter":
                pair.a.update_filter(1, orc.lowpass(2500.0))
                pair.b.update_filter(1, orc.lowpass(2500.0))
            else:
                _, plan = pair.push(x[pos:pos + k * n], 2, shared=(what == "shared"))
                plans.append(plan)
                pos += k * n
    finally:
        pair.close()
    print(f"\nPLANS shared mixed: {plans}")
    assert sum("fused[" in p for p in plans) >= 3, plans


# ---- 5. the largest stream count ------------------------------------------------------------------------------------------
def test_max_stream_count(ctx):
    """65535 streams on one shared row, every stream checked; 65536 streams are still refused at creation."""
    import radiorust_b200 as rr
    import torch

    with pytest.raises(rr.RadiorustError) as e:
        rr.Chain(ctx, [rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(64, 48000.0, 6000.0)], "f32", n_streams=65536)
    assert e.value.code == rr._ffi.RR_ERR_INVALID
    S = 65535
    cfg = down_chain("f32", 960_000.0, 1024, [2, 1, 3, 2], 64, 48000.0, 6000.0, 3000.0)
    x = orc.synth_noise(7500, sum(cfg.pushes) * cfg.n, "f64")
    shifts = class_shifts(cfg.sr)
    ref = references(cfg, x, shifts)
    pair = Pair(ctx, cfg, S, shifts)
    try:
        got, plans = run_pushes(pair, x, 2)
    finally:
        pair.close()
        torch.cuda.empty_cache()
    print(f"\nPLANS shared S={S}: {plans}")
    assert any("fused[" in p or "front+poly2[" in p for p in plans), plans
    check_streams(got, ref, "f32", "streams/65535")


# ---- 6. no replication ---------------------------------------------------------------------------------------------------
def test_no_replication(ctx):
    """C3 with 16384 streams: after a 3-chunk priming push, one shared push of 2^22 samples runs k_fused.  Replicated,
    its input alone would take 550 GB; shared, the free device memory drops by less than an eighth of that (outputs
    and per-stream state).  A seeded sample of 64 streams is checked against the oracle."""
    import torch

    S, n = 16384, 4096
    big = 1 << 22
    esz = 8
    cfg = down_chain("f32", 2_400_000.0, n, [3, big // n], 64, 48000.0, 6000.0, 3000.0)
    total = 3 * n + big
    out_need = S * (total // 50 + 64) * esz
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < out_need + (8 << 30):
        pytest.skip(f"needs {(out_need + (8 << 30)) / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    x = orc.synth_noise(7600, total, "f64")
    shifts = class_shifts(cfg.sr)
    ch = make_chain(ctx, cfg, S, shifts)
    try:
        outs = []
        row, ptr = shared_row(x[:3 * n], "f32", 2)
        cap = ch.max_output(cfg.sr, n, 3)
        y = torch.empty((S, max(cap, 1)), dtype=torch.complex64, device="cuda")
        cnt, _ = ch.push_shared_device(cfg.sr, n, 3, ptr, y.data_ptr(), cap, y.shape[1])
        ch.sync()
        pick = np.sort(np.random.default_rng(7601).choice(S, 64, replace=False))
        pick_d = torch.from_numpy(pick).cuda()
        outs.append(y[pick_d, :cnt].cpu().numpy())
        del y, row
        row, ptr = shared_row(x[3 * n:], "f32", 2)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free0, _ = torch.cuda.mem_get_info()
        cap = ch.max_output(cfg.sr, n, big // n)
        y = torch.empty((S, cap), dtype=torch.complex64, device="cuda")
        cnt, _ = ch.push_shared_device(cfg.sr, n, big // n, ptr, y.data_ptr(), cap, cap)
        ch.sync()
        free1, _ = torch.cuda.mem_get_info()
        plan = ch.plan
        outs.append(y[pick_d, :cnt].cpu().numpy())
        del y, row
    finally:
        ch.close()
        torch.cuda.empty_cache()
    drop = free0 - free1
    print(f"\nSHARED no-replication: plan {plan}, free memory drop {drop / 2**30:.2f} GiB")
    assert "fused[filter+down]" in plan, plan
    assert drop < S * big * esz // 8, drop
    check_streams(np.concatenate(outs, axis=1), references(cfg, x, shifts), "f32", "no-replication", streams=pick)


# ---- 7. refusals ------------------------------------------------------------------------------------------------------------
def test_refusals_leave_the_chain_untouched(ctx, sm, monkeypatch):
    """Null input, a too small out_capacity and an out_stride below the output are refused; the next push then equals
    a twin that never saw the refused call.  A per-stream push with in_stride 0 is still refused."""
    import radiorust_b200 as rr
    import torch

    clear_env(monkeypatch)
    cfg = family("front_poly2")
    S = 2 * K + 3
    n = cfg.n
    x = orc.synth_noise(7700, 16 * n, "f64")
    shifts = class_shifts(cfg.sr)
    pair = Pair(ctx, cfg, S, shifts)
    try:
        pos = 0
        for k in (3, 2):
            pair.push(x[pos:pos + k * n], 2)
            pos += k * n
        k = 2
        cap = pair.a.max_output(cfg.sr, n, k)
        assert cap > 0
        row, ptr = shared_row(x[pos:pos + k * n], "f32", 2)
        y = torch.empty((S, cap + 1), dtype=torch.complex64, device="cuda")
        refusals = [
            (rr._ffi.RR_ERR_INVALID, lambda: pair.a.push_shared_device(cfg.sr, n, k, 0, y.data_ptr(), cap, cap + 1)),
            (rr._ffi.RR_ERR_CAPACITY, lambda: pair.a.push_shared_device(cfg.sr, n, k, ptr, y.data_ptr(), cap - 1, cap + 1)),
            (rr._ffi.RR_ERR_INVALID, lambda: pair.a.push_shared_device(cfg.sr, n, k, ptr, y.data_ptr(), cap, cap - 1)),
            (rr._ffi.RR_ERR_INVALID, lambda: pair.a.push_device(cfg.sr, n, k, ptr, 0, y.data_ptr(), cap, cap + 1)),
            (rr._ffi.RR_ERR_INVALID, lambda: pair.a.push_shared_host_async(cfg.sr, n, k, 0, y.data_ptr(), cap, cap + 1)),
        ]
        for i, (code, call) in enumerate(refusals):
            with pytest.raises(rr.RadiorustError) as e:
                call()
            assert e.value.code == code, (i, e.value)
            # the next push matches the twin that never saw the refused call
            pair.push(x[pos:pos + k * n], 2)
            pos += k * n
    finally:
        pair.close()


# ---- 8. one stream ------------------------------------------------------------------------------------------------------------
def test_single_stream_equals_push(ctx):
    """S = 1: push_shared equals push."""
    cfg = family("front_poly2")
    n = cfg.n
    x = orc.synth_noise(7800, 12 * n, "f64").astype(np.complex64)
    shifts = class_shifts(cfg.sr)
    a = make_chain(ctx, cfg, 1, shifts)
    b = make_chain(ctx, cfg, 1, shifts)
    try:
        pos = 0
        for k in (3, 4, 1, 4):
            ya, ra = a.push_shared(cfg.sr, x[pos:pos + k * n], n)
            yb, rb = b.push(cfg.sr, x[pos:pos + k * n], n)
            assert a.plan == b.plan and ra == rb
            assert np.array_equal(ya, yb)
            pos += k * n
    finally:
        a.close()
        b.close()
