"""Python face of the C ABI: contexts, stage descriptions and the chain.

This is a thin ``ctypes`` layer used by the tests and ``bench.py``; the sample
arithmetic lives in ``csrc/`` (CUDA, sm_100a).  Stage constructors mirror the
reference constructors (names and argument meaning):

=====================  ====================================================
``FreqShifter``        ``blocks::FreqShifter::with_precision_and_shift``  (transform.rs:297)
``Filter``             ``blocks::filters::Filter::{new,new_rectangular,with_window}`` (filters.rs:128-152)
``Downsampler``        ``blocks::Downsampler::with_quality`` (resampling.rs:45)
``Upsampler``          ``blocks::Upsampler::with_quality`` (resampling.rs:180)
``FmDemod``            ``blocks::modulation::FmDemod::new`` (modulation.rs:97)
``GainControl``        ``blocks::GainControl::new`` (transform.rs:43)
``Fourier``            ``blocks::analysis::Fourier::{new,new_center_dc,with_window,with_window_center_dc}`` (analysis.rs:38-59)
=====================  ====================================================
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

from . import _ffi
from ._ffi import check


class Context:
    """One CUDA device (``rr_ctx``)."""

    def __init__(self, device: int = 0):
        self._lib = _ffi.load()
        h = C.c_void_p()
        check(self._lib.rr_ctx_create(device, C.byref(h)))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rr_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # pinned chunk pool at the chain edges (bufferpool.rs:187-222 stand-in)
    def pinned_array(self, shape, dtype) -> np.ndarray:
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        check(self._lib.rr_pinned_alloc(self._h, n, C.byref(p)))
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        return _Pinned(arr, self, p)


class PinnedChunkBufPool:
    """``rr_pool``: recycling pool of pinned host buffers, the chain-edge stand-in for ``ChunkBufPool``
    (bufferpool.rs:187-222).  ``get`` returns a numpy array over a pinned buffer (recycled when one is idle);
    ``put`` is the recycler (``Chunk::drop``, bufferpool.rs:82-90)."""

    def __init__(self, ctx: Context):
        self._lib = _ffi.load()
        self.ctx = ctx
        h = C.c_void_p()
        check(self._lib.rr_pool_create(ctx._h, C.byref(h)))
        self._h = h
        self._loans = {}

    def get(self, shape, dtype) -> np.ndarray:
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        p, cap = C.c_void_p(), C.c_size_t()
        check(self._lib.rr_pool_get(self._h, count * dtype.itemsize, C.byref(p), C.byref(cap)))
        buf = (C.c_char * max(cap.value, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)
        self._loans[arr.ctypes.data] = p.value
        return arr

    def put(self, arr: np.ndarray):
        ptr = self._loans.pop(arr.ctypes.data)
        check(self._lib.rr_pool_put(self._h, C.c_void_p(ptr)))

    def stats(self):
        """(allocated, reused, idle buffers, buffers on loan)"""
        v = [C.c_uint64() for _ in range(4)]
        check(self._lib.rr_pool_stats(self._h, *[C.byref(x) for x in v]))
        return tuple(int(x.value) for x in v)

    def trim(self):
        check(self._lib.rr_pool_trim(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rr_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Pinned(np.ndarray):
    """numpy view of a pinned allocation that frees it when collected."""

    def __new__(cls, arr, ctx, ptr):
        obj = arr.view(cls)
        obj._ctx = ctx
        obj._ptr = ptr
        return obj

    def __array_finalize__(self, obj):
        self._ctx = getattr(obj, "_ctx", None)
        self._ptr = None  # only the original owns the allocation

    def __del__(self):
        if getattr(self, "_ptr", None) is not None and self._ctx is not None and self._ctx._h:
            self._ctx._lib.rr_pinned_free(self._ctx._h, self._ptr)
            self._ptr = None


# ---- stage descriptions ----------------------------------------------------------
@dataclass
class FreqShifter:
    shift: float = 0.0
    precision: float = 1.0


@dataclass
class Filter:
    freq_resp: Callable[[int, float], complex]
    window: Tuple = ("kaiser", math.sqrt(3.0))  # Kaiser::with_null_at_bin(2.0), filters.rs:132

    @classmethod
    def new(cls, freq_resp):
        return cls(freq_resp)

    @classmethod
    def new_rectangular(cls, freq_resp):
        return cls(freq_resp, ("rectangular",))

    @classmethod
    def with_window(cls, freq_resp, window):
        return cls(freq_resp, window)


@dataclass
class Downsampler:
    output_chunk_len: int
    output_rate: float
    bandwidth: float
    quality: float = 3.0


@dataclass
class Upsampler:
    output_chunk_len: int
    output_rate: float
    bandwidth: float
    quality: float = 3.0


@dataclass
class FmDemod:
    deviation: float


@dataclass
class FmMod:
    deviation: float


@dataclass
class Rechunker:
    output_chunk_len: int


@dataclass
class Overlapper:
    chunk_count: int


@dataclass
class GainControl:
    gain: float = 1.0


@dataclass
class Fourier:
    window: Tuple = ("rectangular",)  # Fourier::new (analysis.rs:38-40)
    center_dc: bool = False


def _window_fields(window):
    """-> (kind, beta, ctypes fn or None)"""
    if callable(window):
        cb = _ffi.WINDOW_FN(lambda _u, x: float(window(x)))
        return _ffi.RR_WINDOW_CUSTOM, 0.0, cb
    kind = window[0]
    if kind == "kaiser":
        return _ffi.RR_WINDOW_KAISER, float(window[1]), None
    if kind == "rectangular":
        return _ffi.RR_WINDOW_RECTANGULAR, 0.0, None
    raise ValueError(f"unknown window {window!r}")


def _freq_resp_cb(f):
    def cb(_user, bin_, freq, re, im):
        v = complex(f(int(bin_), float(freq)))
        re[0] = v.real
        im[0] = v.imag

    return _ffi.FREQ_RESP_FN(cb)


class Chain:
    """``rr_chain``: a sequence of blocks run for ``n_streams`` streams in lock step."""

    def __init__(self, ctx: Context, stages: Sequence, dtype: str = "f32", n_streams: int = 1):
        self._lib = _ffi.load()
        self.ctx = ctx
        self.flt = dtype
        self.cdtype = {"f32": np.complex64, "f64": np.complex128}[dtype]
        self.n_streams = int(n_streams)
        self._keep = []  # ctypes callbacks must outlive the chain
        arr = (_ffi.StageDesc * max(len(stages), 1))()
        for i, st in enumerate(stages):
            d = arr[i]
            if isinstance(st, FreqShifter):
                d.kind = _ffi.RR_STAGE_FREQSHIFT
                d.precision = st.precision
                d.shift = st.shift
            elif isinstance(st, Filter):
                d.kind = _ffi.RR_STAGE_FILTER
                cb = _freq_resp_cb(st.freq_resp)
                self._keep.append(cb)
                d.freq_resp = cb
                k, beta, wcb = _window_fields(st.window)
                d.window_kind, d.window_beta = k, beta
                if wcb is not None:
                    self._keep.append(wcb)
                    d.window_fn = wcb
            elif isinstance(st, (Downsampler, Upsampler)):
                d.kind = _ffi.RR_STAGE_DOWNSAMPLE if isinstance(st, Downsampler) else _ffi.RR_STAGE_UPSAMPLE
                d.output_chunk_len = st.output_chunk_len
                d.output_rate = st.output_rate
                d.bandwidth = st.bandwidth
                d.quality = st.quality
            elif isinstance(st, FmDemod):
                d.kind = _ffi.RR_STAGE_FMDEMOD
                d.deviation = st.deviation
            elif isinstance(st, FmMod):
                d.kind = _ffi.RR_STAGE_FMMOD
                d.deviation = st.deviation
            elif isinstance(st, Rechunker):
                d.kind = _ffi.RR_STAGE_RECHUNK
                d.output_chunk_len = st.output_chunk_len
            elif isinstance(st, Overlapper):
                d.kind = _ffi.RR_STAGE_OVERLAP
                d.chunk_count = st.chunk_count
            elif isinstance(st, GainControl):
                d.kind = _ffi.RR_STAGE_GAIN
                d.gain = st.gain
            elif isinstance(st, Fourier):
                d.kind = _ffi.RR_STAGE_FOURIER
                k, beta, wcb = _window_fields(st.window)
                d.window_kind, d.window_beta = k, beta
                if wcb is not None:
                    self._keep.append(wcb)
                    d.window_fn = wcb
                d.center_dc = 1 if st.center_dc else 0
            else:
                raise TypeError(f"not a stage: {st!r}")
        desc = _ffi.ChainDesc()
        desc.dtype = _ffi.RR_C32 if dtype == "f32" else _ffi.RR_C64
        desc.n_streams = self.n_streams
        desc.n_stages = len(stages)
        desc.stages = arr
        h = C.c_void_p()
        check(self._lib.rr_chain_create(ctx._h, C.byref(desc), C.byref(h)))
        self._h = h
        self.stages = list(stages)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rr_chain_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- live parameters (tokio watch channels in the reference) -----------------
    def set_shift(self, stage: int, shift: float, stream: int = -1):
        check(self._lib.rr_chain_set_shift(self._h, stage, stream, float(shift)))

    def set_shifts(self, stage: int, shifts):
        a = np.ascontiguousarray(shifts, dtype=np.float64)
        check(self._lib.rr_chain_set_shifts(self._h, stage, a.ctypes.data_as(C.POINTER(C.c_double)), a.size))

    def shift(self, stage: int, stream: int = 0) -> float:
        v = C.c_double()
        check(self._lib.rr_chain_get_shift(self._h, stage, stream, C.byref(v)))
        return v.value

    def update_filter(self, stage: int, freq_resp, window=None):
        cb = _freq_resp_cb(freq_resp)
        self._keep.append(cb)
        if window is None:
            check(self._lib.rr_chain_update_filter(self._h, stage, cb, None, 0, 0.0, _ffi.WINDOW_FN(), None, 1))
        else:
            k, beta, wcb = _window_fields(window)
            if wcb is not None:
                self._keep.append(wcb)
            check(self._lib.rr_chain_update_filter(self._h, stage, cb, None, k, beta, wcb or _ffi.WINDOW_FN(), None, 0))

    def set_deviation(self, stage: int, deviation: float):
        check(self._lib.rr_chain_set_deviation(self._h, stage, float(deviation)))

    def set_gain(self, stage: int, gain: float):
        check(self._lib.rr_chain_set_gain(self._h, stage, float(gain)))

    def set_output_chunk_len(self, stage: int, output_chunk_len: int):
        check(self._lib.rr_chain_set_output_chunk_len(self._h, stage, int(output_chunk_len)))

    def event(self, is_interrupt: bool = True):
        check(self._lib.rr_chain_event(self._h, 1 if is_interrupt else 0))

    def samples_lost_count(self) -> int:
        """``SamplesLost`` events generated so far by the chain's Rechunker / Overlapper stages."""
        return int(self._lib.rr_chain_samples_lost_count(self._h))

    # ---- data path ------------------------------------------------------------------
    def max_output(self, sample_rate: float, chunk_len: int, n_chunks: int) -> int:
        return int(self._lib.rr_chain_max_output(self._h, float(sample_rate), chunk_len, n_chunks))

    def push(self, sample_rate: float, x: np.ndarray, chunk_len: int, out: Optional[np.ndarray] = None):
        """Push ``x`` ([n_streams, n_chunks*chunk_len] or 1-D for one stream) from HOST memory.

        Returns ``(y, out_rate)`` with ``y`` of shape ``[n_streams, out_count]``.
        """
        x = np.asarray(x)
        if x.ndim == 1:
            x = x[None, :]
        assert x.shape[0] == self.n_streams, "one row per stream"
        assert x.dtype == self.cdtype and x.strides[1] == x.itemsize
        total = x.shape[1]
        assert total % chunk_len == 0
        n_chunks = total // chunk_len if chunk_len else 0
        cap = self.max_output(sample_rate, chunk_len, n_chunks)
        if out is None:
            out = np.empty((self.n_streams, max(cap, 1)), dtype=self.cdtype)
        cnt = C.c_size_t()
        rate = C.c_double()
        check(
            self._lib.rr_chain_push(
                self._h, float(sample_rate), chunk_len, n_chunks, x.ctypes.data, x.strides[0] // x.itemsize,
                out.ctypes.data, out.shape[1], out.strides[0] // out.itemsize, C.byref(cnt), C.byref(rate),
            )
        )
        self.sync()
        return out[:, : cnt.value], rate.value

    def push_device(self, sample_rate, chunk_len, n_chunks, dev_in: int, in_stride: int, dev_out: int, out_capacity: int,
                    out_stride: int):
        """Device-resident push (raw device pointers); returns ``(out_count, out_rate)``; asynchronous."""
        cnt = C.c_size_t()
        rate = C.c_double()
        check(
            self._lib.rr_chain_push_device(
                self._h, float(sample_rate), chunk_len, n_chunks, dev_in, in_stride, dev_out, out_capacity, out_stride,
                C.byref(cnt), C.byref(rate),
            )
        )
        return cnt.value, rate.value

    def push_host_async(self, sample_rate, chunk_len, n_chunks, host_in: int, in_stride: int, host_out: int, out_capacity: int,
                        out_stride: int):
        """``rr_chain_push`` with raw (pinned) host pointers; asynchronous until :meth:`sync`."""
        cnt = C.c_size_t()
        rate = C.c_double()
        check(
            self._lib.rr_chain_push(
                self._h, float(sample_rate), chunk_len, n_chunks, host_in, in_stride, host_out, out_capacity, out_stride,
                C.byref(cnt), C.byref(rate),
            )
        )
        return cnt.value, rate.value

    def push_shared(self, sample_rate: float, x: np.ndarray, chunk_len: int, out: Optional[np.ndarray] = None):
        """Push one 1-D row ``x`` from HOST memory into every stream (``rr_chain_push_shared``): a channelizer tuning all
        its streams out of one wideband input.  Returns ``(y, out_rate)`` with ``y`` of shape ``[n_streams, out_count]``."""
        x = np.asarray(x)
        assert x.ndim == 1, "one row, read by every stream"
        assert x.dtype == self.cdtype and x.strides[0] == x.itemsize
        total = x.shape[0]
        assert total % chunk_len == 0
        n_chunks = total // chunk_len if chunk_len else 0
        cap = self.max_output(sample_rate, chunk_len, n_chunks)
        if out is None:
            out = np.empty((self.n_streams, max(cap, 1)), dtype=self.cdtype)
        cnt = C.c_size_t()
        rate = C.c_double()
        check(
            self._lib.rr_chain_push_shared(
                self._h, float(sample_rate), chunk_len, n_chunks, x.ctypes.data, out.ctypes.data, out.shape[1],
                out.strides[0] // out.itemsize, C.byref(cnt), C.byref(rate),
            )
        )
        self.sync()
        return out[:, : cnt.value], rate.value

    def push_shared_device(self, sample_rate, chunk_len, n_chunks, dev_in: int, dev_out: int, out_capacity: int, out_stride: int):
        """``rr_chain_push_shared_device``: every stream reads the row at ``dev_in`` (raw device pointers); returns
        ``(out_count, out_rate)``; asynchronous."""
        cnt = C.c_size_t()
        rate = C.c_double()
        check(
            self._lib.rr_chain_push_shared_device(
                self._h, float(sample_rate), chunk_len, n_chunks, dev_in, dev_out, out_capacity, out_stride, C.byref(cnt), C.byref(rate),
            )
        )
        return cnt.value, rate.value

    def push_shared_host_async(self, sample_rate, chunk_len, n_chunks, host_in: int, host_out: int, out_capacity: int, out_stride: int):
        """``rr_chain_push_shared`` with raw (pinned) host pointers; asynchronous until :meth:`sync`."""
        cnt = C.c_size_t()
        rate = C.c_double()
        check(
            self._lib.rr_chain_push_shared(
                self._h, float(sample_rate), chunk_len, n_chunks, host_in, host_out, out_capacity, out_stride, C.byref(cnt), C.byref(rate),
            )
        )
        return cnt.value, rate.value

    def copy_out_async(self, dst_dev: int, dst_stride: int, src_dev: int, src_stride: int, n_samples: int):
        """``rr_chain_copy_out_async``: copy-engine copy of a push's outputs (raw device pointers), behind the queued work."""
        check(self._lib.rr_chain_copy_out_async(self._h, dst_dev, dst_stride, src_dev, src_stride, n_samples))

    def sync(self):
        check(self._lib.rr_chain_sync(self._h))

    def set_fast_path(self, enable: bool = True):
        check(self._lib.rr_chain_set_fast_path(self._h, 1 if enable else 0))

    def set_timing(self, enable: bool = True):
        check(self._lib.rr_chain_set_timing(self._h, 1 if enable else 0))

    def kernel_time(self):
        """(total ms, launches, kernel name) of the dominant kernel since ``set_timing(True)``."""
        ms = C.c_double()
        cnt = C.c_int()
        name = C.c_char_p()
        check(self._lib.rr_chain_kernel_time(self._h, C.byref(ms), C.byref(cnt), C.byref(name)))
        return ms.value, cnt.value, (name.value or b"").decode()

    def kernel_breakdown(self):
        """{kernel name: (total ms, launches)} of every timed kernel (call after ``kernel_time``)."""
        out = {}
        for item in self._lib.rr_chain_kernel_breakdown(self._h).decode().split(";"):
            if item:
                name, ms, cnt = item.rsplit(":", 2)
                out[name] = (float(ms), int(cnt))
        return out

    @property
    def cuda_stream(self) -> int:
        return int(self._lib.rr_chain_cuda_stream(self._h) or 0)

    @property
    def plan(self) -> str:
        return self._lib.rr_chain_plan(self._h).decode()


def level(ctx: Context, x: np.ndarray, chunk_len: int) -> np.ndarray:
    """``metering::level`` (metering.rs:21-30) of every chunk of ``x`` ([streams, samples] complex64/128) on the
    device: mean square norm, f64.  Returns [streams, chunks]."""
    lib = _ffi.load()
    x = np.ascontiguousarray(np.atleast_2d(x))
    if x.dtype not in (np.complex64, np.complex128):
        raise TypeError("complex64 or complex128 samples")
    S, total = x.shape
    n_chunks = total // chunk_len if chunk_len else 0
    dev = C.c_void_p()
    check(lib.rr_device_alloc(ctx._h, max(x.nbytes, 16), C.byref(dev)))
    try:
        check(lib.rr_memcpy_h2d(ctx._h, dev, x.ctypes.data_as(C.c_void_p), x.nbytes))
        out = np.zeros((S, n_chunks), dtype=np.float64)
        check(lib.rr_metering_level(ctx._h, _ffi.RR_C32 if x.dtype == np.complex64 else _ffi.RR_C64, dev, total, chunk_len, n_chunks, S,
                                    out.ctypes.data_as(C.POINTER(C.c_double))))
    finally:
        lib.rr_device_free(ctx._h, dev)
    return out


def _with_device_copy(ctx: Context, x: np.ndarray, fn):
    lib = _ffi.load()
    dev = C.c_void_p()
    check(lib.rr_device_alloc(ctx._h, max(x.nbytes, 16), C.byref(dev)))
    try:
        check(lib.rr_memcpy_h2d(ctx._h, dev, x.ctypes.data_as(C.c_void_p), x.nbytes))
        return fn(lib, dev)
    finally:
        lib.rr_device_free(ctx._h, dev)


def _bins_2d(bins: np.ndarray) -> np.ndarray:
    bins = np.ascontiguousarray(np.atleast_2d(bins))
    if bins.dtype not in (np.complex64, np.complex128):
        raise TypeError("complex64 or complex128 samples")
    return bins


def bandwidth(ctx: Context, double_percentile: float, sample_rate: float, bins: np.ndarray, chunk_len: int) -> np.ndarray:
    """``metering::bandwidth`` (metering.rs:42-84) of every chunk of Fourier-transformed ``bins``
    ([streams, samples]) on the device.  Returns hertz, [streams, chunks]."""
    bins = _bins_2d(bins)
    S, total = bins.shape
    n_chunks = total // chunk_len if chunk_len else 0
    out = np.zeros((S, n_chunks), dtype=np.float64)

    def run(lib, dev):
        check(lib.rr_metering_bandwidth(ctx._h, _ffi.RR_C32 if bins.dtype == np.complex64 else _ffi.RR_C64, dev, total, chunk_len, n_chunks,
                                        S, float(double_percentile), float(sample_rate), out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    return _with_device_copy(ctx, bins, run)


def rescale_energy(ctx: Context, resolution: int, bins: np.ndarray, chunk_len: int) -> np.ndarray:
    """``metering::rescale_energy`` (metering.rs:93-110) of every chunk of ``bins`` on the device.
    Returns [streams, chunks, resolution] in the real type of ``bins``."""
    bins = _bins_2d(bins)
    S, total = bins.shape
    n_chunks = total // chunk_len if chunk_len else 0
    out = np.zeros((S, n_chunks, resolution), dtype=np.float32 if bins.dtype == np.complex64 else np.float64)

    def run(lib, dev):
        check(lib.rr_metering_rescale_energy(ctx._h, _ffi.RR_C32 if bins.dtype == np.complex64 else _ffi.RR_C64, dev, total, chunk_len,
                                             n_chunks, S, int(resolution), out.ctypes.data_as(C.c_void_p)))
        return out

    return _with_device_copy(ctx, bins, run)


def kernel_launch_count() -> int:
    return int(_ffi.load().rr_kernel_launch_count())
