"""Device-resident pushes at the layouts callers use, with every stream checked against the f64 oracle.

The kernels see the caller's base pointer and ``in_stride`` only on a device push (a host push is first compacted into
staging buffers), so the layouts here are pushed through ``rr_chain_push_device``: windows of a larger buffer, padded
and odd strides, a base one sample off a 16-byte boundary, padded output strides.  The last two turn ``tma_ok`` off
for f32, and the chain then routes to other kernels; the tests assert which.

Many streams, every one checked: the chain is linear for a fixed shift, so stream s is built on the device as
``x_s = a_s*A + b_s*B`` (seeded complex weights of order 1, two shared base signals) and gets shift class ``s mod K``.
K is coprime to the SM count, so the stream a persistent CTA processes just before s (stride ``gridDim.x``) has another
shift and other weights: state leaking from one stream into the next changes the output.  The f64 oracle runs once per
(class, base signal); stream s must come out as ``a_s*ref(A, k) + b_s*ref(B, k)``.  (For f32 chains the device rounds
``x_s`` to f32: about 6e-8 relative, far below the bounds.)

Bounds, asserted per stream (never pooled over streams).  rel = ||y - ref|| / ||ref||, max = max_m |y - ref| / rms(ref):

    =====  =======  =======  ======================================================================================
    type   rel      max      why
    =====  =======  =======  ======================================================================================
    f32    3e-6     3e-5     the f32 oracle itself sits at 2.5e-7 ... 1.1e-6 rel and 6e-7 ... 9e-6 max against
                             the f64 oracle (C3 4.1e-7 / 2.0e-6, C1 3.0e-7 / 1.6e-6, P = 20 3.4e-7 / 1.4e-6,
                             C2 1250/3 1.1e-6 / 9.1e-6, Filter 2n = 2^15 2.5e-7 / 9.4e-7, Upsampler x50 7e-8 / 6.1e-7)
    f64    1e-12    1e-11
    =====  =======  =======  ======================================================================================

Worst per-stream values measured on a B200 (148 SMs, 1000 W power limit), over every layout and stream of each case:

    ==============================================  =======  =======
    case (plan)                                     rel      max
    ==============================================  =======  =======
    fused P = 20 / 40 / 50 (fused[...])             3.9e-7   2.0e-6
    front+poly2 (C3, 17 streams)                    3.7e-7   1.7e-6
    front+poly, k_front<16> (C1 64/3)               3.5e-7   1.4e-6
    front+poly, k_front_wide (75/2)                 3.7e-7   1.3e-6
    poly, f64 (C3)                                  1.2e-15  4.2e-15
    fused_os (fast path off)                        6.3e-7   1.8e-6
    big_os, 2n = 2^15, f32 / f64 (k_long_*)         7.0e-7   2.8e-6  /  1.3e-15  4.9e-15
    upsample x50 (k_upsample_phase) / x3 (tiled)    7.0e-8   7.6e-7
    rechunk(view) -> nco+poly2                      3.0e-7   9.2e-7
    overlap -> fused_os[filter]                     3.6e-7   1.7e-6
    stream counts SM-1 ... 3 SM+5, and 65535        3.9e-7   1.6e-6
    rows 2^30 samples apart, f32 / f64              3.1e-7   1.1e-6  /  1.2e-15  3.7e-15
    NCO edges (fused, front+poly2, front+poly,      6.9e-7   2.7e-6
    fused_os)
    ==============================================  =======  =======
"""
import math

import numpy as np
import pytest

from oracle import radiorust_oracle as orc

pytestmark = pytest.mark.gpu

BOUNDS = {"f32": (3e-6, 3e-5), "f64": (1e-12, 1e-11)}
K = 7  # shift classes; coprime to the SM count (asserted)


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


# ---- inputs and reference -----------------------------------------------------------------------------------------
def weights(S, seed):
    rng = np.random.default_rng(seed)
    w = (0.5 + rng.random((2, S))) * np.exp(2j * np.pi * rng.random((2, S)))
    return w[0], w[1]


class Inputs:
    """Base signals A, B (f64, host and device) and the weights of S streams."""

    def __init__(self, S, total, seed):
        import torch

        self.S = S
        self.A = orc.synth_noise(seed, total, "f64")
        self.B = orc.synth_noise(seed + 1, total, "f64")
        self.a, self.b = weights(S, seed + 2)
        self.A_d, self.B_d = (torch.from_numpy(v).cuda() for v in (self.A, self.B))
        self.a_d, self.b_d = (torch.from_numpy(v).cuda() for v in (self.a, self.b))

    def fill(self, view, lo, dtype):
        """view[s, :] = a_s*A[lo:lo+w] + b_s*B[lo:lo+w] (view: [S, w] device tensor of any strides)."""
        w = view.shape[1]
        blk = max(1, (1 << 25) // max(w, 1))
        for s0 in range(0, self.S, blk):
            s1 = min(self.S, s0 + blk)
            view[s0:s1] = (self.a_d[s0:s1, None] * self.A_d[None, lo:lo + w] + self.b_d[s0:s1, None] * self.B_d[None, lo:lo + w]).to(dtype)


def oracle_run(blocks, sr, x, n, retune=None):
    """The oracle fed chunk by chunk; retune = (chunk index, stage, shift): set_shift before that chunk."""
    chain = orc.Chain(blocks)
    outs = []
    for c in range(len(x) // n):
        if retune is not None and c == retune[0]:
            blocks[retune[1]].set_shift(retune[2])
        outs += [m.chunk for m in chain.push(orc.Samples(sr, x[c * n:(c + 1) * n])) if isinstance(m, orc.Samples)]
    return np.concatenate(outs) if outs else np.zeros(0, np.complex128)


def references(cfg, inp, shifts, retune_shifts=None):
    """[K, M] f64 oracle outputs of A and of B per shift class (one row when the chain has no FreqShifter)."""
    ra, rb = [], []
    for k in range(K if cfg.nco is not None else 1):
        for base, out in ((inp.A, ra), (inp.B, rb)):
            rt = None if retune_shifts is None else (cfg.retune_chunk, cfg.nco, retune_shifts[k])
            out.append(oracle_run(cfg.oracle(shifts[k] if cfg.nco is not None else 0.0), cfg.sr, base, cfg.n, rt))
    return np.stack(ra), np.stack(rb)


def check_streams(got, inp, ra, rb, flt, label):
    """Every stream against a_s*ref(A, s mod K) + b_s*ref(B, s mod K); returns (worst rel, worst max)."""
    S, M = got.shape
    assert S == inp.S and M == ra.shape[1] and M > 0, (got.shape, ra.shape)
    lim_rel, lim_max = BOUNDS[flt]
    rel = np.empty(S)
    mx = np.empty(S)
    for s0 in range(0, S, 4096):
        s1 = min(S, s0 + 4096)
        cls = np.arange(s0, s1) % ra.shape[0]
        want = inp.a[s0:s1, None] * ra[cls] + inp.b[s0:s1, None] * rb[cls]
        err = got[s0:s1].astype(np.complex128) - want
        den = np.linalg.norm(want, axis=1)
        rel[s0:s1] = np.linalg.norm(err, axis=1) / den
        mx[s0:s1] = np.abs(err).max(axis=1) / (den / math.sqrt(M))
    bad = np.flatnonzero(~((rel <= lim_rel) & (mx <= lim_max)))
    wr, wm = float(np.nanmax(rel)), float(np.nanmax(mx))
    print(f"\nLAYOUT {label}: {flt} streams={S} outputs={M} worst rel {wr:.2e} max {wm:.2e}")
    assert bad.size == 0, (label, f"{bad.size} of {S} streams out of bounds, first {bad[:8].tolist()}",
                           rel[bad[:8]].tolist(), mx[bad[:8]].tolist())
    return wr, wm


# ---- chains ---------------------------------------------------------------------------------------------------------
class Cfg:
    """One chain: GPU stages, f64 oracle blocks for a shift, push sizes, the plan it must take.

    nco: index of the FreqShifter stage (None: no FreqShifter).  plan: substring of the plan of some push of the
    contiguous run.  tma_plan: for f32 chains whose kernels need a 16-byte aligned base and an even stride, the
    substring the other layouts' plans must contain instead (None: the same plans as the contiguous run)."""

    def __init__(self, flt, sr, n, pushes, gpu, oracle, nco=0, plan="", tma_plan=None, not_tma=(), precision=1.0,
                 fast_path=True, retune_chunk=None):
        self.flt, self.sr, self.n, self.pushes = flt, sr, n, list(pushes)
        self.gpu, self.oracle, self.nco = gpu, oracle, nco
        self.plan, self.tma_plan, self.not_tma = plan, tma_plan, not_tma
        self.precision, self.fast_path, self.retune_chunk = precision, fast_path, retune_chunk


def down_chain(flt, sr, n, pushes, ocl, out_rate, bw, cutoff, precision=1.0, **kw):
    """FreqShifter -> Filter(low-pass) -> Downsampler."""
    import radiorust_b200 as rr

    return Cfg(flt, sr, n, pushes,
               lambda: [rr.FreqShifter(0.0, precision), rr.Filter.new(orc.lowpass(cutoff)), rr.Downsampler(ocl, out_rate, bw)],
               lambda shift: [orc.FreqShifter("f64", precision, shift), orc.Filter.new("f64", orc.lowpass(cutoff)),
                              orc.Downsampler("f64", ocl, out_rate, bw)], precision=precision, **kw)


def family(name):
    import radiorust_b200 as rr

    TMA = dict(tma_plan="poly[filter+down]", not_tma=("front", "fused["))
    if name in ("fused_p20", "fused_p40", "fused_p50"):
        sr, n, ocl, bw = {"fused_p20": (960_000.0, 2048, 17, 20000.0), "fused_p40": (1_920_000.0, 4096, 64, 6000.0),
                          "fused_p50": (2_400_000.0, 4096, 64, 6000.0)}[name]
        return down_chain("f32", sr, n, [3, 5, 4, 6], ocl, 48000.0, bw, bw / 2, plan="fused[filter+down]", **TMA)
    if name == "front_poly2":    # C3 below the k_fused stream count
        return down_chain("f32", 2_400_000.0, 4096, [3, 5, 2, 6], 64, 48000.0, 6000.0, 3000.0, plan="front+poly2[filter+down]", **TMA)
    if name == "front16_poly":   # C1, P/Q = 64/3: k_front<16> + k_poly on u
        return down_chain("f32", 1_024_000.0, 4096, [3, 10, 1, 2, 5], 192, 48000.0, 6000.0, 3000.0, plan="front+poly[filter+down]",
                          tma_plan="poly[filter+down]", not_tma=("front",))
    if name == "front_wide_poly":  # P/Q = 75/2: k_front_wide reads any layout
        return down_chain("f32", 1_200_000.0, 4096, [2, 9, 4], 100, 32000.0, 6000.0, 3000.0, plan="front+poly[filter+down]")
    if name == "poly_f64":       # C3 in f64: k_poly on all branches
        return down_chain("f64", 2_400_000.0, 4096, [3, 10, 5], 50, 48000.0, 6000.0, 3000.0, plan="poly[filter+down]")
    if name == "fused_os":       # the stateful overlap-save kernel with the decimating epilogue
        return down_chain("f32", 2_400_000.0, 4096, [2, 3, 1], 64, 48000.0, 6000.0, 3000.0, plan="fused_os[filter+down]", fast_path=False)
    if name in ("long_f32", "long_f64"):  # 2n = 2^15: the streaming four-step kernels (k_long_*)
        flt = name[-3:]
        return Cfg(flt, 2_400_000.0, 16384, [1, 2, 1], lambda: [rr.Filter.new(orc.lowpass(20000.0))],
                   lambda _s: [orc.Filter.new("f64", orc.lowpass(20000.0))], nco=None, plan="big_os")
    if name == "upsample_x50":   # 11 taps per phase: k_upsample_phase
        return Cfg("f32", 48000.0, 1024, [1, 3, 2, 2], lambda: [rr.Upsampler(4096, 2_400_000.0, 20000.0)],
                   lambda _s: [orc.Upsampler("f64", 4096, 2_400_000.0, 20000.0)], nco=None, plan="upsample")
    if name == "upsample_x3":    # the tiled kernel
        return Cfg("f32", 16000.0, 2048, [1, 3, 2, 2], lambda: [rr.Upsampler(4096, 48000.0, 7000.0)],
                   lambda _s: [orc.Upsampler("f64", 4096, 48000.0, 7000.0)], nco=None, plan="upsample")
    if name == "rechunk_view":   # the next stages read the caller's buffer under the new chunk length (n = 1024: k_poly2)
        return Cfg("f32", 2_400_000.0, 4096, [2, 3, 5, 4],
                   lambda: [rr.Rechunker(1024), rr.FreqShifter(0.0), rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(64, 48000.0, 6000.0)],
                   lambda shift: [orc.Rechunker(1024), orc.FreqShifter("f64", 1.0, shift), orc.Filter.new("f64", orc.lowpass(3000.0)),
                                  orc.Downsampler("f64", 64, 48000.0, 6000.0)], nco=1, plan="rechunk(view)", **TMA)
    if name == "overlap":
        return Cfg("f32", 48000.0, 512, [1, 3, 2, 1], lambda: [rr.Overlapper(2), rr.Filter.new(orc.lowpass(5000.0))],
                   lambda _s: [orc.Overlapper(2), orc.Filter.new("f64", orc.lowpass(5000.0))], nco=None, plan="overlap")
    raise KeyError(name)


def class_shifts(sr):
    return [float(round(sr * f)) for f in (1 / 7, -1 / 3, 0.0, 0.0514, -0.2404, 0.4, -0.45)]


# ---- device pushes --------------------------------------------------------------------------------------------------
LAYOUTS = {
    "contiguous": {},
    "pad_even": {"in_pad": 6},
    "odd_stride": {"in_pad": 3},
    "base_plus_1": {"base": 1},
    "windows": {"windows": True},        # every push a window of one [S, total] buffer (in_stride = total > len)
    "out_pad": {"out_pad": 37},
}
TMA_OFF = ("odd_stride", "base_plus_1")  # an 8-byte f32 sample: misaligned rows / base


def make_chain(ctx, cfg, S, shifts):
    import radiorust_b200 as rr

    ch = rr.Chain(ctx, cfg.gpu(), cfg.flt, n_streams=S)
    if cfg.nco is not None:
        ch.set_shifts(cfg.nco, [shifts[s % K] for s in range(S)])
    if not cfg.fast_path:
        ch.set_fast_path(False)
    return ch


def device_push(ch, cfg, inp, layout, row_stride=None, retune=None):
    """Lay the streams out as `layout` says and push cfg.pushes windows in sequence; returns ([S, M] host outputs,
    plan of every push).  Padding around the pushed samples holds NaN: nothing outside [0, len) of a row may be read.
    row_stride (windows only): distance of the streams' rows.  retune = (push index, shifts per stream)."""
    import torch

    S, n = inp.S, cfg.n
    cdt = torch.complex64 if cfg.flt == "f32" else torch.complex128
    esz = 8 if cfg.flt == "f32" else 16
    base, in_pad, out_pad = layout.get("base", 0), layout.get("in_pad", 0), layout.get("out_pad", 0)
    total = sum(cfg.pushes) * n
    whole = None
    if layout.get("windows"):
        stride = row_stride or total
        whole = torch.empty(base + (S - 1) * stride + total, dtype=cdt, device="cuda")
        view = whole.as_strided((S, total), (stride, 1), base)
        inp.fill(view, 0, cdt)
    outs, plans, pos = [], [], 0
    for i, k in enumerate(cfg.pushes):
        if retune is not None and i == retune[0]:
            ch.set_shifts(cfg.nco, retune[1])
        L = k * n
        if whole is not None:
            ptr = view.data_ptr() + pos * n * esz
        else:
            stride = L + in_pad
            buf = torch.full((base + S * stride,), float("nan"), dtype=cdt, device="cuda")
            v = buf.as_strided((S, L), (stride, 1), base)
            inp.fill(v, pos * n, cdt)
            ptr = v.data_ptr()
        cap = ch.max_output(cfg.sr, n, k)
        ostride = cap + out_pad
        y = torch.full((max(S * ostride, 1),), float("nan"), dtype=cdt, device="cuda")
        torch.cuda.synchronize()
        cnt, _ = ch.push_device(cfg.sr, n, k, ptr, stride, y.data_ptr(), cap, ostride)
        ch.sync()
        outs.append(y.as_strided((S, cnt), (ostride, 1)).cpu().numpy())
        plans.append(ch.plan)
        pos += k
        del y
    del whole
    return np.concatenate(outs, axis=1), plans


# ---- 1. layout sweep ------------------------------------------------------------------------------------------------
FAMILIES = ["fused_p20", "fused_p40", "fused_p50", "front_poly2", "front16_poly", "front_wide_poly", "poly_f64", "fused_os",
            "long_f32", "long_f64", "upsample_x50", "upsample_x3", "rechunk_view", "overlap"]


@pytest.mark.parametrize("name", FAMILIES)
def test_layout_sweep(ctx, sm, monkeypatch, name):
    """Every layout of LAYOUTS through one path family, every stream against the f64 oracle.  Layouts that take the
    same plans as the contiguous run must give bit-identical outputs; where tma_ok is off another plan runs and must be
    correct too.  The k_fused families run at the default stream threshold (2 per SM), the others below it."""
    for v in ("RR_FUSED_MIN_STREAMS", "RR_DISABLE_FUSED", "RR_DISABLE_FRONT", "RR_DISABLE_POLY", "RR_DISABLE_POLY2"):
        monkeypatch.delenv(v, raising=False)
    cfg = family(name)
    S = 2 * sm + 3 if name.startswith("fused_p") else 2 * K + 3
    inp = Inputs(S, sum(cfg.pushes) * cfg.n, 4100 + FAMILIES.index(name) * 10)
    shifts = class_shifts(cfg.sr)
    ra, rb = references(cfg, inp, shifts)
    first = None
    for lname, layout in LAYOUTS.items():
        ch = make_chain(ctx, cfg, S, shifts)
        got, plans = device_push(ch, cfg, inp, layout)
        ch.close()
        print(f"\nPLANS {name} {lname}: {plans}")
        check_streams(got, inp, ra, rb, cfg.flt, f"{name}/{lname}")
        if first is None:
            first = (got, plans)
            assert any(cfg.plan in p for p in plans), plans
            continue
        if cfg.flt == "f32" and cfg.tma_plan is not None and lname in TMA_OFF:
            assert plans != first[1], plans
            assert any(cfg.tma_plan in p for p in plans), plans
            assert not any(bad in p for p in plans for bad in cfg.not_tma), plans
        else:
            assert plans == first[1], (lname, plans, first[1])
            assert np.array_equal(got, first[0]), lname


# ---- 2. stream counts around the k_fused grid --------------------------------------------------------------------
@pytest.mark.parametrize("mult,add,force", [(2, 0, False), (2, 1, False), (3, 5, False), (1, -1, True), (1, 0, True), (1, 1, True)])
def test_stream_counts_around_the_fused_grid(ctx, sm, monkeypatch, mult, add, force):
    """k_fused walks streams with the stride min(S, SMs): stream counts at and around the grid's size, at the default
    threshold and forced.  Push sizes of 1 ... 5 chunks change the front end's live tiles per stream (and so the
    rotation of the tiles over its warps from one stream to the next); after the first two pushes every push is
    steady state and runs k_fused."""
    monkeypatch.delenv("RR_DISABLE_FUSED", raising=False)
    if force:
        monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    else:
        monkeypatch.delenv("RR_FUSED_MIN_STREAMS", raising=False)
    S = mult * sm + add
    cfg = down_chain("f32", 2_400_000.0, 4096, [2, 1, 2, 3, 1, 5, 2, 1, 4], 64, 48000.0, 6000.0, 3000.0)
    inp = Inputs(S, sum(cfg.pushes) * cfg.n, 5200)
    shifts = class_shifts(cfg.sr)
    ra, rb = references(cfg, inp, shifts)
    ch = make_chain(ctx, cfg, S, shifts)
    got, plans = device_push(ch, cfg, inp, LAYOUTS["contiguous"])
    ch.close()
    print(f"\nPLANS S={S}: {plans}")
    assert "front+poly2[" in plans[1] and all("fused[" in p for p in plans[2:]), plans
    check_streams(got, inp, ra, rb, "f32", f"streams/{S}")


# ---- 3. the largest stream count ------------------------------------------------------------------------------------
def test_max_stream_count(ctx):
    """65535 streams (the grid's y limit) on a C3-like chain with P = 20, every stream checked; 65536 are refused."""
    import radiorust_b200 as rr
    import torch

    with pytest.raises(rr.RadiorustError) as e:
        rr.Chain(ctx, [rr.Filter.new(orc.lowpass(3000.0)), rr.Downsampler(64, 48000.0, 6000.0)], "f32", n_streams=65536)
    assert e.value.code == rr._ffi.RR_ERR_INVALID
    S = 65535
    cfg = down_chain("f32", 960_000.0, 1024, [2, 1, 3, 2], 64, 48000.0, 6000.0, 3000.0, plan="front+poly2[filter+down]")
    inp = Inputs(S, sum(cfg.pushes) * cfg.n, 5300)
    shifts = class_shifts(cfg.sr)
    ra, rb = references(cfg, inp, shifts)
    ch = make_chain(ctx, cfg, S, shifts)
    got, plans = device_push(ch, cfg, inp, LAYOUTS["windows"])
    ch.close()
    print(f"\nPLANS S={S}: {plans}")
    assert any("fused[" in p or "front+poly2[" in p for p in plans), plans
    check_streams(got, inp, ra, rb, "f32", "streams/65535")
    del inp
    torch.cuda.empty_cache()


# ---- 4. sample offsets past 2^31 -----------------------------------------------------------------------------------
@pytest.mark.parametrize("flt", ["f32", "f64"])
def test_stream_rows_past_2_31_samples(ctx, monkeypatch, flt):
    """Three streams 2^30 samples apart: stream 2 starts at sample 2^31 of the caller's buffer (32-bit sample
    index arithmetic would wrap).  f32 runs k_front + k_poly2 and then k_fused, f64 k_poly."""
    import torch

    monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    monkeypatch.delenv("RR_DISABLE_FUSED", raising=False)
    S, row = 3, 1 << 30
    cfg = down_chain(flt, 2_400_000.0, 4096, [3, 4, 5], 64, 48000.0, 6000.0, 3000.0)
    esz = 8 if flt == "f32" else 16
    need = ((S - 1) * row + sum(cfg.pushes) * cfg.n) * esz
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < need + (2 << 30):
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    inp = Inputs(S, sum(cfg.pushes) * cfg.n, 5400)
    shifts = class_shifts(cfg.sr)
    ra, rb = references(cfg, inp, shifts)
    ch = make_chain(ctx, cfg, S, shifts)
    try:
        got, plans = device_push(ch, cfg, inp, LAYOUTS["windows"], row_stride=row)
    finally:
        ch.close()
        torch.cuda.empty_cache()
    print(f"\nPLANS rows 2^30 {flt}: {plans}")
    if flt == "f32":
        assert "front+poly2[" in plans[0] and all("fused[" in p for p in plans[1:]), plans
    else:
        assert all("poly[filter+down]" in p for p in plans), plans
    check_streams(got, inp, ra, rb, flt, f"rows2^30/{flt}")


# ---- 5. NCO edges -----------------------------------------------------------------------------------------------
FINE_DENOM = 1_073_741_827  # a prime above 2^30: the ratio of every nonzero shift keeps it as its denominator


def nco_case(name, variant):
    sr = 1_024_000.0 if name == "front16_poly" else 2_400_000.0
    if variant == "fine":   # precision sr / FINE_DENOM: table index and products near 2^30 ... 2^61
        precision = sr / FINE_DENOM
        shifts = [sr / 2 - 3.0, -(sr / 2 - 2.0), -sr / 2, -123456.789, 1.5, -0.25, sr / 2 - 0.5]
        retune = [-v for v in shifts]
    else:                   # precision 1 Hz, reduced denominators <= 32000: the table index wraps several times
        precision = 1.0
        fr = [(1, 2), (-1, 2), (15999, 32000), (-7, 32000), (3, 8), (-3999, 8000), (1, 4)]
        shifts = [sr * p / q for p, q in fr]
        retune = [sr * p / q for p, q in [(-1, 4), (7, 32000), (-1, 2), (3999, 8000), (1, 2), (-15999, 32000), (-3, 8)]]
    pushes = [3, 6, 6, 1, 6, 6]
    common = dict(precision=precision, retune_chunk=sum(pushes[:4]))
    if name == "front16_poly":
        cfg = down_chain("f32", sr, 4096, pushes, 192, 48000.0, 6000.0, 3000.0, plan="front+poly[filter+down]", **common)
    else:
        cfg = down_chain("f32", sr, 4096, pushes, 64, 48000.0, 6000.0, 3000.0, fast_path=(name != "fused_os"),
                         plan={"fused": "fused[", "front_poly2": "front+poly2[", "fused_os": "fused_os["}[name], **common)
    return cfg, shifts, retune


@pytest.mark.parametrize("variant", ["fine", "wrap"])
@pytest.mark.parametrize("name", ["fused", "front_poly2", "front16_poly", "fused_os"])
def test_nco_edges(ctx, monkeypatch, name, variant):
    """Shifts within a few hertz of +-sr/2 and negative ones, a precision whose table has >= 2^30 entries, tables
    that wrap several times within the run, and a retune of every stream between two pushes."""
    monkeypatch.delenv("RR_FUSED_MIN_STREAMS", raising=False)
    monkeypatch.delenv("RR_DISABLE_FUSED", raising=False)
    if name == "fused":
        monkeypatch.setenv("RR_FUSED_MIN_STREAMS", "1")
    elif name == "front_poly2":
        monkeypatch.setenv("RR_DISABLE_FUSED", "1")
    cfg, shifts, retune = nco_case(name, variant)
    total = sum(cfg.pushes) * cfg.n
    for v in shifts + retune:
        num, den = orc.freq_to_ratio(cfg.sr, cfg.precision, v)
        if variant == "fine":
            assert num == 0 or den >= 1 << 30, (v, num, den)
        else:
            assert 3 * den <= total, (v, den)
    S = 2 * K
    inp = Inputs(S, total, 5500 + 10 * len(name) + len(variant))
    ra, rb = references(cfg, inp, shifts, retune)
    ch = make_chain(ctx, cfg, S, shifts)
    got, plans = device_push(ch, cfg, inp, LAYOUTS["windows"], retune=(4, [retune[s % K] for s in range(S)]))
    ch.close()
    print(f"\nPLANS nco {name} {variant}: {plans}")
    assert sum(cfg.plan in p for p in plans) >= 3, plans
    check_streams(got, inp, ra, rb, "f32", f"nco/{name}/{variant}")
