"""Summed-output pushes: every stream's output of a push added into one row (rr_chain_push_summed[_device]).

A transmit channelizer moves n_streams baseband channels onto their carriers and adds them into the wideband row of one
SDR.  The row is defined from the per-stream outputs alone: out[t] = sum over s ascending of y_s[t], each y_s[t] what a
per-stream push writes (already rounded to Flt), added in f64 from +0.0 and rounded once.  Two checks:

- twin, bit for bit: a second chain with the same configuration takes rr_chain_push_device of the same rows; its rows
  are added on the host in that order (complex128, a Python loop over s) and rounded to the chain's dtype.  The summed
  row must equal that bit for bit, and the samples behind out_count (NaN sentinels) must survive.  The summed plan is
  the twin's with "upsample|freqshift" replaced by "synth[upsample+nco+sum]" (k_synth), or with "|sum" appended
  (k_stream_sum); every case asserts which.
- oracle: Upsampler -> FreqShifter is linear.  Stream s is a_s*A + b_s*B with shift class s mod K, so the expected row
  is sum_c (sum_{s in c} a_s) Y_{A,c} + (sum_{s in c} b_s) Y_{B,c}: 2K f64 oracle runs whatever S is.

Oracle bound, per sample (a sum of many carriers cancels, so a relative L2 norm of the row says nothing):

    |row[t] - want[t]| <= 32 * eps_T * sum_s E_s[t],   E_s[t] = sum_p |x_s[p]| |h[t - p*Q]|,

E_s the magnitude envelope of stream s's interpolation (|y_s[t]| <= E_s[t]; the mixer has unit gain).  Bounded by
|a_s| E_A + |b_s| E_B, computed with scipy's upfirdn from the f64 taps.  Per stream and sample, with u = eps_T / 2:
the input rounded to Flt and the Flt taps, 2u E; the NT <= 16 fma's of a phase, NT u E; the NCO phase
start + i/denom*tau in Flt (|phase| < 3 pi: the quotient, tau and the sum rounded), < 22u; sin/cos, 2u; the complex
product, 2u; all times E.  The f64 sum adds S * 2^-53 relative, the final rounding u |row| <= u sum_s E_s.  At most
(16 + 2 + 22 + 2 + 2 + 1) u = 45u < 64u = 32 eps_T.
"""
import math

import numpy as np
import pytest

from oracle import radiorust_oracle as orc
from test_gpu_layout import K, class_shifts, oracle_run

pytestmark = pytest.mark.gpu

SYNTH = "synth[upsample+nco+sum]"


@pytest.fixture(scope="module")
def ctx():
    import radiorust_b200 as rr

    c = rr.Context(0)
    yield c
    c.close()


def cdtype(flt):
    import torch

    return (torch.complex64, np.complex64) if flt == "f32" else (torch.complex128, np.complex128)


def summed_plan(plan, fused):
    if fused:
        assert "upsample|freqshift" in plan, plan
        return plan.replace("upsample|freqshift", SYNTH)
    return plan + "|sum"


def host_sum(rows, flt):
    """rows [S, M] -> the contract's row: complex128 from +0.0, streams ascending, rounded once."""
    acc = np.zeros(rows.shape[1], np.complex128)
    for s in range(rows.shape[0]):
        acc += rows[s].astype(np.complex128)
    return acc.astype(cdtype(flt)[1])


def bits(v):
    return v.view(np.uint32 if v.dtype == np.complex64 else np.uint64)


def make_chain(ctx, stages, flt, S, nco, shifts):
    import radiorust_b200 as rr

    ch = rr.Chain(ctx, stages(), flt, n_streams=S)
    if nco is not None:
        ch.set_shifts(nco, [shifts[s % K] for s in range(S)])
    return ch


def device_rows(x, flt, lead=1, pad=3):
    """x [S, L] (host) as device rows with NaN on both sides; returns (buffer, ptr, stride)."""
    import torch

    cdt, npdt = cdtype(flt)
    S, L = x.shape
    stride = L + lead + pad
    buf = torch.full((S * stride + lead,), float("nan"), dtype=cdt, device="cuda")
    v = buf.as_strided((S, L), (stride, 1), lead)
    v[:] = torch.from_numpy(np.ascontiguousarray(x.astype(npdt))).cuda()
    return buf, v.data_ptr(), stride


class Pair:
    """Chain a takes summed pushes, its twin b per-stream pushes of the same rows."""

    def __init__(self, ctx, stages, flt, S, nco=None, shifts=None, sr=48000.0, fused=True):
        self.flt, self.S, self.sr, self.fused = flt, S, sr, fused
        self.a = make_chain(ctx, stages, flt, S, nco, shifts)
        self.b = make_chain(ctx, stages, flt, S, nco, shifts)

    def close(self):
        self.a.close()
        self.b.close()

    def push(self, x, n, summed=True):
        """One push of x [S, k*n] to both; asserts the row, the sentinels and the plan.  summed=False gives a a
        per-stream push too (rows compared with b's).  Returns (row or rows, plan)."""
        import torch

        S, flt = self.S, self.flt
        k = x.shape[1] // n
        cdt, _ = cdtype(flt)
        cap = self.a.max_output(self.sr, n, k)
        assert cap == self.b.max_output(self.sr, n, k)
        buf, ptr, stride = device_rows(x, flt)
        ostride = cap + 1
        yb = torch.full((max(S * ostride, 1),), float("nan"), dtype=cdt, device="cuda")
        ya = torch.full((cap + 8,), float("nan"), dtype=cdt, device="cuda") if summed else torch.full_like(yb, float("nan"))
        torch.cuda.synchronize()
        if summed:
            ca, ra = self.a.push_summed_device(self.sr, n, k, ptr, stride, ya.data_ptr(), cap)
        else:
            ca, ra = self.a.push_device(self.sr, n, k, ptr, stride, ya.data_ptr(), cap, ostride)
        cb, rb = self.b.push_device(self.sr, n, k, ptr, stride, yb.data_ptr(), cap, ostride)
        self.a.sync()
        self.b.sync()
        assert ca == cb and (ca == 0 or ra == rb), (ca, cb, ra, rb)
        gb = yb.as_strided((S, cb), (ostride, 1)).cpu().numpy()
        if not summed:
            assert self.a.plan == self.b.plan
            assert np.array_equal(bits(ya.as_strided((S, ca), (ostride, 1)).cpu().numpy()), bits(gb))
            return gb, self.a.plan
        got = ya.cpu().numpy()
        assert np.isnan(got[ca:]).all(), "samples behind out_count were written"
        want = host_sum(gb, flt)
        assert np.array_equal(bits(got[:ca]), bits(want)), f"summed row differs from the sum of the twin's rows ({self.a.plan})"
        if ca > 0:
            assert self.a.plan == summed_plan(self.b.plan, self.fused), (self.a.plan, self.b.plan)
        else:
            assert self.a.plan == self.b.plan, (self.a.plan, self.b.plan)  # nothing emitted, nothing summed
        return got[:ca], self.a.plan


# ---- chains ------------------------------------------------------------------------------------------------------------
def fm_up50():
    """A TX channel: FmMod -> Upsampler x50 (L = 515, 11 taps per phase) -> FreqShifter."""
    import radiorust_b200 as rr

    return [rr.FmMod(5000.0), rr.Upsampler(4096, 2_400_000.0, 20000.0), rr.FreqShifter(0.0)]


def stages_of(name):
    import radiorust_b200 as rr

    return {
        "fm_up50_f32": fm_up50,
        "fm_up50_f64": fm_up50,
        "up8_nt4": lambda: [rr.Upsampler(1000, 384000.0, 24000.0, 1.0), rr.FreqShifter(0.0)],      # L = 32: 4 taps per phase
        "up256_nt16": lambda: [rr.Upsampler(50000, 2_048_000.0, 4500.0), rr.FreqShifter(0.0)],     # L = 3511: 14 taps per phase
        "up3_tiled": lambda: [rr.Upsampler(4096, 48000.0, 7000.0), rr.FreqShifter(0.0)],
        "up_indexed": lambda: [rr.Upsampler(2048, 96000.0, 20000.0), rr.FreqShifter(0.0)],
        "fmmod_nco": lambda: [rr.FmMod(5000.0), rr.FreqShifter(0.0)],
        "rx_down": lambda: [rr.FreqShifter(0.0), rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(64, 48000.0, 6000.0)],
        "fourier_last": lambda: [rr.FreqShifter(0.0), rr.Fourier()],
    }[name]


# name: (dtype, input rate, FreqShifter's rate, chunk length, pushes, FreqShifter stage, k_synth route)
FAMILIES = {
    "fm_up50_f32": ("f32", 48000.0, 2_400_000.0, 1024, [1, 3, 2, 2], 2, True),
    "fm_up50_f64": ("f64", 48000.0, 2_400_000.0, 1024, [1, 3, 2, 2], 2, True),
    "up8_nt4": ("f32", 48000.0, 384000.0, 512, [2, 1, 3, 5], 1, True),
    "up256_nt16": ("f32", 8000.0, 2_048_000.0, 256, [2, 3, 1, 4], 1, True),
    "up3_tiled": ("f32", 16000.0, 48000.0, 2048, [1, 3, 2], 1, False),
    "up_indexed": ("f32", 48000.5, 96000.0, 1024, [1, 3, 2], 1, False),
    "fmmod_nco": ("f64", 48000.0, 48000.0, 512, [1, 3, 2], 1, False),
    "rx_down": ("f32", 2_400_000.0, 2_400_000.0, 4096, [3, 5, 2], 0, False),
    "fourier_last": ("f32", 48000.0, 48000.0, 1024, [1, 3, 2], 0, False),
}
PLANS = {"up3_tiled": "upsample|freqshift|sum", "up_indexed": "upsample(indexed)|freqshift|sum", "fmmod_nco": "fmmod|freqshift|sum",
         "rx_down": "[filter+down]|sum", "fourier_last": "freqshift|fourier|sum"}


def family_pair(ctx, name, S):
    flt, sr, nco_rate, n, pushes, nco, fused = FAMILIES[name]
    return Pair(ctx, stages_of(name), flt, S, nco, class_shifts(nco_rate), sr, fused)


def noise_rows(S, total, seed, flt):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((S, total)) + 1j * rng.standard_normal((S, total))) / math.sqrt(2)
    return x.astype(cdtype(flt)[1])


# ---- 1. twin, every family ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(FAMILIES))
def test_twin_bit_for_bit(ctx, name):
    flt, sr, _, n, pushes, _, fused = FAMILIES[name]
    S = 2 * K + 3
    x = noise_rows(S, sum(pushes) * n, 8100 + list(FAMILIES).index(name), flt)
    pair = family_pair(ctx, name, S)
    plans, pos = [], 0
    try:
        for k in pushes:
            row, plan = pair.push(x[:, pos:pos + k * n], n)
            plans.append(plan)
            pos += k * n
    finally:
        pair.close()
    print(f"\nPLANS summed {name}: {plans}")
    if fused:
        assert any(SYNTH in p for p in plans), plans
        assert not any("|sum" in p for p in plans), plans
    else:
        assert any(p.endswith(PLANS[name]) for p in plans), plans


# ---- 2. push sequences on the fused route -----------------------------------------------------------------------------------
def test_push_sequences_and_state(ctx):
    """Chunks of 64 inputs give 3200 outputs against output chunks of 4096: pushes that emit nothing, samples pending
    across pushes, 1 to 5 chunks per push; retunes, deviation changes, interrupt events, and per-stream pushes on the
    summed chain, each step against the twin."""
    S, n = 2 * K + 3, 64
    shifts = class_shifts(2_400_000.0)
    pair = Pair(ctx, fm_up50, "f32", S, 2, shifts)
    x = noise_rows(S, 64 * n, 8200, "f32")
    retune = [-shifts[(s + 3) % K] / 2 for s in range(S)]
    steps = [("sum", 1), ("sum", 2), ("sum", 5), ("sum", 1), ("retune", 0), ("sum", 3), ("per_stream", 2), ("sum", 4),
             ("deviation", 0), ("sum", 1), ("sum", 1), ("event", 0), ("sum", 5), ("per_stream", 1), ("sum", 2), ("sum", 3)]
    plans, counts, pos = [], [], 0
    try:
        for what, k in steps:
            if what == "retune":
                pair.a.set_shifts(2, retune)
                pair.b.set_shifts(2, retune)
            elif what == "deviation":
                pair.a.set_deviation(0, 7500.0)
                pair.b.set_deviation(0, 7500.0)
            elif what == "event":
                pair.a.event(True)
                pair.b.event(True)
            else:
                out, plan = pair.push(x[:, pos:pos + k * n], n, summed=(what == "sum"))
                plans.append(plan)
                counts.append(out.shape[-1])
                pos += k * n
    finally:
        pair.close()
    print(f"\nPLANS summed sequence: {list(zip(plans, counts))}")
    assert 0 in counts and sum(SYNTH in p for p in plans) >= 8, (plans, counts)


# ---- 3. the linear-combination oracle ------------------------------------------------------------------------------------
def tx_cfg(flt):
    import radiorust_b200 as rr

    return (lambda: [rr.Upsampler(4096, 2_400_000.0, 20000.0), rr.FreqShifter(0.0)],
            lambda shift: [orc.Upsampler("f64", 4096, 2_400_000.0, 20000.0), orc.FreqShifter("f64", 1.0, shift)])


def envelope(x, M):
    """E[t] = sum_p |x[p]| |h[t - 50 p]| of the x50 Upsampler (f64 taps), t < M."""
    from scipy.signal import upfirdn

    up = orc.Upsampler("f64", 4096, 2_400_000.0, 20000.0)
    up._design(48000.0)
    e = upfirdn(np.abs(up.ir), np.abs(x), up=50)
    out = np.zeros(M)
    out[:min(M, len(e))] = e[:M]
    return out


def check_oracle(row, A, B, a, b, shifts, flt, t0=0, label=""):
    """row[i] (absolute sample t0 + i) against the linear combination of the 2K class references; inputs A, B cover
    the push from sample 0."""
    _, oracle = tx_cfg(flt)
    M = t0 + len(row)
    S = len(a)
    cls = np.arange(S) % K
    want = np.zeros(len(row), np.complex128)
    for c in range(K):
        for base, w in ((A, a), (B, b)):
            y = oracle_run(oracle(shifts[c]), 48000.0, base, len(base))
            assert len(y) >= M, (len(y), M)
            want += w[cls == c].sum() * y[t0:M]
    env = (np.abs(a).sum() * envelope(A, M) + np.abs(b).sum() * envelope(B, M))[t0:]
    eps = np.finfo(np.float32 if flt == "f32" else np.float64).eps
    err = np.abs(row.astype(np.complex128) - want)
    ratio = err / (eps * env)
    print(f"\nSUMMED oracle {label}: {flt} streams={S} samples={len(row)} worst err/(eps*sum E) {ratio.max():.2f}")
    assert (err <= 32 * eps * env).all(), (label, int(np.argmax(ratio)), float(ratio.max()))


@pytest.mark.parametrize("flt", ["f32", "f64"])
def test_oracle_linear_combination(ctx, flt):
    import torch

    from test_gpu_layout import Inputs

    S, n, k = 3 * K + 2, 1024, 6
    inp = Inputs(S, n * k, 8300 + (flt == "f64"))
    stages, _ = tx_cfg(flt)
    shifts = class_shifts(2_400_000.0)
    ch = make_chain(ctx, stages, flt, S, 1, shifts)
    cdt, _ = cdtype(flt)
    try:
        x = torch.empty((S, n * k), dtype=cdt, device="cuda")
        inp.fill(x, 0, cdt)
        cap = ch.max_output(48000.0, n, k)
        y = torch.full((cap + 4,), float("nan"), dtype=cdt, device="cuda")
        cnt, _ = ch.push_summed_device(48000.0, n, k, x.data_ptr(), x.shape[1], y.data_ptr(), cap)
        ch.sync()
        assert ch.plan == SYNTH, ch.plan
        row = y[:cnt].cpu().numpy()
    finally:
        ch.close()
    check_oracle(row, inp.A, inp.B, inp.a, inp.b, shifts, flt, label=flt)


# ---- 4. beyond per-stream memory ------------------------------------------------------------------------------------------
def test_beyond_per_stream_memory(ctx):
    """8192 streams x 2^17 inputs at x50: per-stream outputs would take 430 GB, the summed row is 52 MB.  The row's
    first 2^18 samples and its last ones (from 2 s in, where every shift's NCO is back at phase 0) are checked
    against the oracle."""
    import torch

    from test_gpu_layout import Inputs

    S, total = 8192, 1 << 17
    need = S * total * 8 + (2 << 30)
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    inp = Inputs(S, total, 8400)
    stages, _ = tx_cfg("f32")
    shifts = class_shifts(2_400_000.0)
    ch = make_chain(ctx, stages, "f32", S, 1, shifts)
    try:
        x = torch.empty((S, total), dtype=torch.complex64, device="cuda")
        inp.fill(x, 0, torch.complex64)
        cap = ch.max_output(48000.0, total, 1)
        y = torch.full((cap + 4,), float("nan"), dtype=torch.complex64, device="cuda")
        free0, _ = torch.cuda.mem_get_info()
        cnt, _ = ch.push_summed_device(48000.0, total, 1, x.data_ptr(), total, y.data_ptr(), cap)
        ch.sync()
        free1, _ = torch.cuda.mem_get_info()
        plan = ch.plan
        row = y.cpu().numpy()
        del x, y
    finally:
        ch.close()
        torch.cuda.empty_cache()
    print(f"\nSUMMED beyond memory: plan {plan}, {cnt} samples, free memory drop {(free0 - free1) / 2**30:.2f} GiB")
    assert plan == SYNTH, plan
    assert np.isnan(row[cnt:]).all()
    assert free0 - free1 < (1 << 30)
    head = 1 << 18
    check_oracle(row[:head], inp.A[:head // 50 + 16], inp.B[:head // 50 + 16], inp.a, inp.b, shifts, "f32", label="head")
    p0 = 96000  # 2 s: every class shift is an integer number of hertz, so each NCO is back at its start phase
    tail_in = slice(p0, total)
    # the oracle run on the inputs from p0 gives the outputs from t = 50*p0; the first 16*50 of them miss the inputs in
    # front of p0, and the oracle emits whole chunks only
    t_skip = 16 * 50
    seg = row[p0 * 50 + t_skip:p0 * 50 + 1_700_000]
    check_oracle(seg, inp.A[tail_in], inp.B[tail_in], inp.a, inp.b, shifts, "f32", t0=t_skip, label="tail")


# ---- 5. edges ----------------------------------------------------------------------------------------------------------------
def test_single_stream_is_the_per_stream_push(ctx):
    """S = 1: the summed row is the per-stream push's output, bit for bit, on both routes."""
    for name in ("fm_up50_f32", "up3_tiled"):
        flt, sr, nco_rate, n, pushes, nco, _ = FAMILIES[name]
        x = noise_rows(1, sum(pushes) * n, 8500, flt)
        a = make_chain(ctx, stages_of(name), flt, 1, nco, class_shifts(nco_rate))
        b = make_chain(ctx, stages_of(name), flt, 1, nco, class_shifts(nco_rate))
        try:
            pos = 0
            for k in pushes:
                ya, ra = a.push_summed(sr, x[:, pos:pos + k * n], n)
                yb, rb = b.push(sr, x[:, pos:pos + k * n], n)
                assert ra == rb and np.array_equal(bits(ya), bits(yb[0]))
                pos += k * n
        finally:
            a.close()
            b.close()


@pytest.mark.parametrize("name", ["fm_up50_f32", "fmmod_nco"])
def test_max_stream_count(ctx, name):
    """65535 streams, small pushes (64 inputs: 3200 outputs per stream at x50), on each route."""
    import torch

    S, n = 65535, 64
    pair = family_pair(ctx, name, S)
    x = noise_rows(S, 4 * n, 8600, FAMILIES[name][0])
    try:
        plans = [pair.push(x[:, :2 * n], n)[1], pair.push(x[:, 2 * n:], n)[1]]
    finally:
        pair.close()
        torch.cuda.empty_cache()
    print(f"\nPLANS summed S={S} {name}: {plans}")
    assert (SYNTH in plans[-1]) == FAMILIES[name][6], plans


def test_host_equals_device(ctx):
    """push_summed (host rows) equals push_summed_device bit for bit; then three push_summed_host_async calls back to
    back from pinned buffers with one sync."""
    import torch

    flt, sr, _, n, _, nco, _ = FAMILIES["fm_up50_f32"]
    S = 2 * K + 3
    shifts = class_shifts(2_400_000.0)
    pushes = [1, 3, 2, 4, 1, 3]
    x = noise_rows(S, sum(pushes) * n, 8700, flt)
    host = make_chain(ctx, fm_up50, flt, S, nco, shifts)
    dev = make_chain(ctx, fm_up50, flt, S, nco, shifts)
    try:
        def dev_push(xs, k):
            cap = dev.max_output(sr, n, k)
            buf, ptr, stride = device_rows(xs, flt)
            y = torch.full((cap + 1,), float("nan"), dtype=torch.complex64, device="cuda")
            torch.cuda.synchronize()
            cnt, _ = dev.push_summed_device(sr, n, k, ptr, stride, y.data_ptr(), cap)
            dev.sync()
            return y[:cnt].cpu().numpy()

        pos = 0
        for k in pushes[:3]:
            yh, _ = host.push_summed(sr, x[:, pos:pos + k * n], n)
            yd = dev_push(x[:, pos:pos + k * n], k)
            assert host.plan == dev.plan and SYNTH in host.plan and np.array_equal(bits(yh), bits(yd))
            pos += k * n
        pins, outs, counts = [], [], []
        for k in pushes[3:]:
            pin = ctx.pinned_array((S, k * n), np.complex64)
            pin[:] = x[:, pos:pos + k * n]
            cap = host.max_output(sr, n, k)
            pout = ctx.pinned_array((cap + 1,), np.complex64)
            pout[:] = np.nan
            cnt, _ = host.push_summed_host_async(sr, n, k, pin.ctypes.data, k * n, pout.ctypes.data, cap)
            pins.append(pin)
            outs.append(pout)
            counts.append(cnt)
            pos += k * n
        host.sync()
        pos = sum(pushes[:3]) * n
        for k, pout, cnt in zip(pushes[3:], outs, counts):
            yd = dev_push(x[:, pos:pos + k * n], k)
            assert np.array_equal(bits(np.asarray(pout[:cnt])), bits(yd)) and np.isnan(pout[cnt:]).all()
            pos += k * n
    finally:
        host.close()
        dev.close()


# ---- 6. refusals ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["fm_up50_f32", "up3_tiled"])
def test_refusals_leave_the_chain_untouched(ctx, name):
    """A row too small (RR_ERR_CAPACITY), null pointers and in_stride < len (RR_ERR_INVALID) are refused; the next push
    still matches the twin."""
    import radiorust_b200 as rr
    import torch

    flt, sr, _, n, _, _, _ = FAMILIES[name]
    S = 2 * K + 3
    pair = family_pair(ctx, name, S)
    x = noise_rows(S, 16 * n, 8800, flt)
    try:
        pos = 0
        pair.push(x[:, :3 * n], n)
        pos = 3 * n
        k = 2
        cap = pair.a.max_output(sr, n, k)
        assert cap > 0
        buf, ptr, stride = device_rows(x[:, pos:pos + k * n], flt)
        y = torch.empty((cap,), dtype=cdtype(flt)[0], device="cuda")
        a = pair.a
        refusals = [
            (rr._ffi.RR_ERR_CAPACITY, lambda: a.push_summed_device(sr, n, k, ptr, stride, y.data_ptr(), cap - 1)),
            (rr._ffi.RR_ERR_INVALID, lambda: a.push_summed_device(sr, n, k, 0, stride, y.data_ptr(), cap)),
            (rr._ffi.RR_ERR_INVALID, lambda: a.push_summed_device(sr, n, k, ptr, stride, 0, cap)),
            (rr._ffi.RR_ERR_INVALID, lambda: a.push_summed_device(sr, n, k, ptr, k * n - 1, y.data_ptr(), cap)),
            (rr._ffi.RR_ERR_INVALID, lambda: a.push_summed_host_async(sr, n, k, 0, k * n, y.data_ptr(), cap)),
        ]
        for i, (code, call) in enumerate(refusals):
            with pytest.raises(rr.RadiorustError) as e:
                call()
            assert e.value.code == code, (i, e.value)
            pair.push(x[:, pos:pos + k * n], n)
            pos += k * n
    finally:
        pair.close()
