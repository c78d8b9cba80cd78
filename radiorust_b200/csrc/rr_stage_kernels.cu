// Stand-alone stage kernels: NCO/mixer, gain, FIR decimator, zero-stuffing
// interpolator, FM discriminator, strided copy.  Used when a chain cannot be
// fused (large FFTs, long resampler kernels, FM chains) and as the reference
// implementation of each stage on the device.  sm_100a.
#include <algorithm>

#include "rr_chain_os.cuh"

namespace rr {

// Element-wise pass over one stream: every thread keeps kMapUnroll independent 8/16-byte loads in flight
// (coalesced: consecutive threads, consecutive samples) before it stores; f(t, sample) -> sample.
constexpr int kMapUnroll = 4;
template <typename T, typename F>
__device__ __forceinline__ void map_stream(const cx<T>* __restrict__ src, cx<T>* __restrict__ dst, long long len, F f) {
    const long long tile = (long long)blockDim.x * kMapUnroll;
    for (long long t0 = (long long)blockIdx.x * tile + threadIdx.x; t0 < len; t0 += (long long)gridDim.x * tile) {
        cx<T> v[kMapUnroll];
#pragma unroll
        for (int u = 0; u < kMapUnroll; ++u) {
            const long long t = t0 + (long long)u * blockDim.x;
            if (t < len) v[u] = ld_cx(&src[t]);
        }
#pragma unroll
        for (int u = 0; u < kMapUnroll; ++u) {
            const long long t = t0 + (long long)u * blockDim.x;
            if (t < len) st_cx(&dst[t], f(t, v[u]));
        }
    }
}
// CTAs along x for `len` samples per stream when the grid's y dimension runs over n_streams streams
inline unsigned map_grid_x(long long len, int n_streams) {
    long long bx = (len + 256 * kMapUnroll - 1) / (256 * kMapUnroll);
    const long long cap = std::max<long long>(1, (1LL << 16) / std::max(1, n_streams));  // ~64 K CTAs in all
    if (bx > cap) bx = cap;
    if (bx > 4096) bx = 4096;
    return (unsigned)bx;
}

// ---------------------------------------------------------------------------
// FreqShifter hot loop, src/blocks/transform.rs:341-348, with phase_vec[idx]
// (transform.rs:333-338) evaluated on the fly from the integer recurrence.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_freqshift(const cx<T>* __restrict__ in, long long in_stride,
                                                   cx<T>* __restrict__ out, long long out_stride, long long len,
                                                   const NcoStream* __restrict__ nco, long long nco_offset) {
    const int s = blockIdx.y;
    const NcoStream ns = nco[s];
    const cx<T>* src = in + (long long)s * in_stride;
    cx<T>* dst = out + (long long)s * out_stride;
    const T start = (T)ns.start_phase;
    map_stream<T>(src, dst, len, [&](long long t, cx<T> v) {
        const uint32_t k = (uint32_t)(((unsigned long long)ns.idx + (unsigned long long)(nco_offset + t)) % ns.denom);
        const uint32_t i = mulmod_u32(ns.numer_abs, k, ns.denom);
        return cmul(v, nco_phasor<T>(i, ns.denom, ns.sign, start));
    });
}

__global__ void k_nco_advance(NcoStream* nco, int n_streams, long long len) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n_streams) {
        const NcoStream ns = nco[s];
        nco[s].idx = (uint32_t)(((unsigned long long)ns.idx + (unsigned long long)len) % ns.denom);
    }
}

cudaError_t launch_nco_advance(NcoStream* nco, int n_streams, long long len, cudaStream_t st) {
    k_nco_advance<<<(n_streams + 127) / 128, 128, 0, st>>>(nco, n_streams, len);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_freqshift(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                             int n_streams, const NcoStream* nco, long long nco_offset, cudaStream_t st) {
    if (len <= 0) return cudaSuccess;
    dim3 grid(map_grid_x(len, n_streams), (unsigned)n_streams);
    k_freqshift<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<cx<T>*>(out),
                                         out_stride, len, nco, nco_offset);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// GainControl, src/blocks/transform.rs:60-62
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_gain(const cx<T>* __restrict__ in, long long in_stride, cx<T>* __restrict__ out,
                                              long long out_stride, long long len, T gain) {
    const int s = blockIdx.y;
    const cx<T>* src = in + (long long)s * in_stride;
    cx<T>* dst = out + (long long)s * out_stride;
    map_stream<T>(src, dst, len, [&](long long, cx<T> v) { return cscale(v, gain); });
}
template <typename T>
cudaError_t launch_gain(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                        int n_streams, double gain, cudaStream_t st) {
    if (len <= 0) return cudaSuccess;
    dim3 grid(map_grid_x(len, n_streams), (unsigned)n_streams);
    k_gain<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<cx<T>*>(out),
                                    out_stride, len, (T)gain);
    return cudaGetLastError();
}

template <typename T>
__global__ void __launch_bounds__(256) k_copy2d(const cx<T>* __restrict__ in, long long in_stride,
                                                cx<T>* __restrict__ out, long long out_stride, long long len) {
    const int s = blockIdx.y;
    const cx<T>* src = in + (long long)s * in_stride;
    cx<T>* dst = out + (long long)s * out_stride;
    map_stream<T>(src, dst, len, [](long long, cx<T> v) { return v; });
}
template <typename T>
cudaError_t launch_copy2d(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                          int n_streams, cudaStream_t st) {
    if (len <= 0) return cudaSuccess;
    dim3 grid(map_grid_x(len, n_streams), (unsigned)n_streams);
    k_copy2d<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<cx<T>*>(out),
                                      out_stride, len);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Downsampler hot loop, src/blocks/resampling.rs:103-121: one warp per output
// sample, window over [tail | input].
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_downsample(const cx<T>* __restrict__ in, long long in_stride, long long len,
                                                    const cx<T>* __restrict__ tail_in, const T* __restrict__ ir, int L,
                                                    RateState rate, long long n_out, cx<T>* __restrict__ out,
                                                    long long out_stride) {
    const int s = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const long long o = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (o >= n_out) return;
    const cx<T>* src = in + (long long)s * in_stride;
    const cx<T>* tl = tail_in + (long long)s * (L - 1);
    const long long m = rate.m0 + 1 + o;
    const long long jm = (m * rate.P + rate.Q - 1) / rate.Q;
    const long long first = jm - rate.j0 - L;  // index (in this push) of the oldest window sample
    T ax = (T)0, ay = (T)0;
    for (int t = lane; t < L; t += 32) {
        const long long idx = first + t;
        const cx<T> z = (idx < 0) ? ld_cx(&tl[(L - 1) + idx]) : ld_cx(&src[idx]);
        const T h = ir[t];
        ax = fma(z.x, h, ax);
        ay = fma(z.y, h, ay);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        ax += __shfl_xor_sync(0xffffffffu, ax, d);
        ay += __shfl_xor_sync(0xffffffffu, ay, d);
    }
    if (lane == 0) st_cx(&out[(long long)s * out_stride + o], cx<T>(ax, ay));
}

// The same with the firing instants from a table (rates that are not integer valued: the reference's f64 `pos`
// recurrence, replayed on the host): output o ends at input sample fire[o] of this push.
template <typename T>
__global__ void __launch_bounds__(256) k_downsample_idx(const cx<T>* __restrict__ in, long long in_stride, const cx<T>* __restrict__ tail_in,
                                                        const T* __restrict__ ir, int L, const int* __restrict__ fire, long long n_out,
                                                        cx<T>* __restrict__ out, long long out_stride) {
    const int s = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const long long o = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (o >= n_out) return;
    const cx<T>* src = in + (long long)s * in_stride;
    const cx<T>* tl = tail_in + (long long)s * (L - 1);
    const long long first = (long long)fire[o] - L + 1;  // index (in this push) of the oldest window sample
    T ax = (T)0, ay = (T)0;
    for (int t = lane; t < L; t += 32) {
        const long long idx = first + t;
        const cx<T> z = (idx < 0) ? ld_cx(&tl[(L - 1) + idx]) : ld_cx(&src[idx]);
        const T h = ir[t];
        ax = fma(z.x, h, ax);
        ay = fma(z.y, h, ay);
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        ax += __shfl_xor_sync(0xffffffffu, ax, d);
        ay += __shfl_xor_sync(0xffffffffu, ay, d);
    }
    if (lane == 0) st_cx(&out[(long long)s * out_stride + o], cx<T>(ax, ay));
}

// new tail = last L-1 samples of [tail_in | input]
template <typename T>
__global__ void k_tail_update(const cx<T>* __restrict__ in, long long in_stride, long long len,
                              const cx<T>* __restrict__ tail_in, cx<T>* __restrict__ tail_out, int L) {
    const int s = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= L - 1) return;
    const long long pos = len - (L - 1) + i;
    const cx<T> v = (pos < 0) ? ld_cx(&tail_in[(long long)s * (L - 1) + (L - 1) + pos])
                              : ld_cx(&in[(long long)s * in_stride + pos]);
    st_cx(&tail_out[(long long)s * (L - 1) + i], v);
}

template <typename T>
cudaError_t launch_downsample(const void* in, long long in_stride, long long len, const void* tail_in, void* tail_out,
                              const T* ir, int L, RateState rate, long long n_out, void* out, long long out_stride,
                              int n_streams, cudaStream_t st) {
    if (n_out > 0) {
        dim3 grid((unsigned)((n_out + 7) / 8), (unsigned)n_streams);
        k_downsample<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len,
                                              reinterpret_cast<const cx<T>*>(tail_in), ir, L, rate, n_out,
                                              reinterpret_cast<cx<T>*>(out), out_stride);
    }
    if (L > 1) {
        dim3 grid((unsigned)((L - 1 + 127) / 128), (unsigned)n_streams);
        k_tail_update<T><<<grid, 128, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len,
                                               reinterpret_cast<const cx<T>*>(tail_in),
                                               reinterpret_cast<cx<T>*>(tail_out), L);
    }
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_downsample_indexed(const void* in, long long in_stride, long long len, const void* tail_in, void* tail_out, const T* ir, int L,
                                      const int* fire, long long n_out, void* out, long long out_stride, int n_streams, cudaStream_t st) {
    if (n_out > 0) {
        dim3 grid((unsigned)((n_out + 7) / 8), (unsigned)n_streams);
        k_downsample_idx<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<const cx<T>*>(tail_in), ir, L, fire,
                                                  n_out, reinterpret_cast<cx<T>*>(out), out_stride);
    }
    if (L > 1) {
        dim3 grid((unsigned)((L - 1 + 127) / 128), (unsigned)n_streams);
        k_tail_update<T><<<grid, 128, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len, reinterpret_cast<const cx<T>*>(tail_in),
                                               reinterpret_cast<cx<T>*>(tail_out), L);
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// Upsampler, src/blocks/resampling.rs:238-267 in gather form: output q is the
// carried partial sum plus sum_p x[p]*ir[q - q_p] over this push's inputs with
// q_p = ceil(p*Q/P) in (q-L, q], accumulated in input order like the ring.
// Outputs q >= m1 are the new carried partial sums.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_upsample(const cx<T>* __restrict__ in, long long in_stride, long long len,
                                                  const cx<T>* __restrict__ acc_in, cx<T>* __restrict__ acc_out,
                                                  const T* __restrict__ ir, int L, RateState rate, long long n_out,
                                                  cx<T>* __restrict__ out, long long out_stride) {
    const int s = blockIdx.y;
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // output index relative to m0
    if (o >= n_out + L) return;
    const long long P = rate.P, Q = rate.Q;  // in/out = P/Q
    const long long q = rate.m0 + o;
    const cx<T>* src = in + (long long)s * in_stride;
    cx<T> acc = (o < L) ? ld_cx(&acc_in[(long long)s * L + o]) : cx<T>((T)0, (T)0);
    // inputs p (global index) with ceil(p*Q/P) <= q  <=>  p <= floor(q*P/Q)
    long long p_hi, p_lo;
    if (P == 1 && q < (1LL << 31) && Q < (1LL << 31)) {  // 32-bit divisions are several times cheaper
        const uint32_t q32 = (uint32_t)q, Q32 = (uint32_t)Q;
        p_hi = q32 / Q32;
        p_lo = (q - L < 0) ? rate.j0 : (long long)((q32 - (uint32_t)L) / Q32) + 1;
    } else {
        p_hi = (q * P) / Q;
        p_lo = (q - L < 0) ? rate.j0 : ((q - L) * P) / Q + 1;
    }
    if (p_lo < rate.j0) p_lo = rate.j0;
    if (p_hi > rate.j0 + len - 1) p_hi = rate.j0 + len - 1;
    if (P == 1) {
        // integer interpolation factor (q_p = p*Q): the tap index walks in steps of Q, no division per tap.  Same
        // order of accumulation (p ascending) as the general loop below.
        long long t = q - p_lo * Q;  // tap of input p_lo, decreasing by Q per input
        for (long long p = p_lo; p <= p_hi; ++p, t -= Q) {
            if (t >= 0 && t < L) {
                const cx<T> x = ld_cx(&src[p - rate.j0]);
                const T h = ir[t];
                acc.x = fma(x.x, h, acc.x);
                acc.y = fma(x.y, h, acc.y);
            }
        }
    } else {
        for (long long p = p_lo; p <= p_hi; ++p) {
            const long long qp = (p * Q + P - 1) / P;
            const int t = (int)(q - qp);
            if (t >= 0 && t < L) {
                const cx<T> x = ld_cx(&src[p - rate.j0]);
                const T h = ir[t];
                acc.x = fma(x.x, h, acc.x);
                acc.y = fma(x.y, h, acc.y);
            }
        }
    }
    if (o < n_out) st_cx(&out[(long long)s * out_stride + o], acc);
    else st_cx(&acc_out[(long long)s * L + (o - n_out)], acc);
}

// Integer interpolation factors (in/out = 1/Q, e.g. 48 kS/s -> 2.4 MS/s), tiled: a CTA takes UP_TILE consecutive outputs
// of one stream, brings the inputs they depend on and the taps into shared memory once, and every thread then walks its
// outputs' ~L/Q taps from there.  Same sums in the same order as k_upsample (inputs ascending, resampling.rs:239-246);
// the general kernel spends most of its time on 64-bit index arithmetic and dependent global loads per tap.
constexpr int UP_TILE = 2048;
template <typename T>
__global__ void __launch_bounds__(256) k_upsample_tiled(const cx<T>* __restrict__ in, long long in_stride, long long len,
                                                        const cx<T>* __restrict__ acc_in, cx<T>* __restrict__ acc_out,
                                                        const T* __restrict__ ir, int L, int Q, long long j0, long long m0, long long n_out,
                                                        cx<T>* __restrict__ out, long long out_stride, int x_cap, cx<T>* __restrict__ out2,
                                                        long long out2_stride, long long out_split) {
    extern __shared__ __align__(16) unsigned char up_smem[];
    T* irs = reinterpret_cast<T*>(up_smem);                                   // [L]
    cx<T>* xs = reinterpret_cast<cx<T>*>(irs + ((L + 1) & ~1));                // [x_cap]
    const int s = blockIdx.y;
    const long long o0 = (long long)blockIdx.x * UP_TILE;
    const long long total = n_out + L;
    const long long o1 = min(o0 + UP_TILE, total);
    const cx<T>* src = in + (long long)s * in_stride;
    // inputs (global index p) that reach outputs [o0, o1): q_p = p*Q in (q - L, q]
    const long long q_first = m0 + o0, q_last = m0 + o1 - 1;
    long long p_lo = (q_first - L < 0) ? 0 : (q_first - L) / Q + 1;
    long long p_hi = q_last / Q;
    if (p_lo < j0) p_lo = j0;
    if (p_hi > j0 + len - 1) p_hi = j0 + len - 1;
    const int n_x = (int)max(0LL, p_hi - p_lo + 1);
    for (int i = threadIdx.x; i < L; i += blockDim.x) irs[i] = ir[i];
    for (int i = threadIdx.x; i < n_x; i += blockDim.x) xs[i] = ld_cx(&src[p_lo - j0 + i]);
    __syncthreads();
    for (long long o = o0 + threadIdx.x; o < o1; o += blockDim.x) {
        const long long q = m0 + o;
        cx<T> acc = (o < L) ? ld_cx(&acc_in[(long long)s * L + o]) : cx<T>((T)0, (T)0);
        long long a_lo = (q - L < 0) ? 0 : (q - L) / Q + 1, a_hi = q / Q;
        if (a_lo < p_lo) a_lo = p_lo;
        if (a_hi > p_hi) a_hi = p_hi;
        int t = (int)(q - a_lo * Q);       // tap of input a_lo, decreasing by Q per input
        int xi = (int)(a_lo - p_lo);
        for (long long p = a_lo; p <= a_hi; ++p, t -= Q, ++xi) {
            if (t >= 0 && t < L) {
                const cx<T> x = xs[xi];
                const T h = irs[t];
                acc.x = fma(x.x, h, acc.x);
                acc.y = fma(x.y, h, acc.y);
            }
        }
        if (o < n_out) {
            // optional second destination: outputs from out_split on belong behind the last whole output chunk
            if (out2 != nullptr && o >= out_split) st_cx(&out2[(long long)s * out2_stride + (o - out_split)], acc);
            else st_cx(&out[(long long)s * out_stride + o], acc);
        } else {
            st_cx(&acc_out[(long long)s * L + (o - n_out)], acc);
        }
    }
}

// Integer interpolation factors, one output PHASE per thread: output q = p*Q + r is sum_k ir[r + k*Q] * x[p - k],
// k < NT = ceil(L / Q).  Thread (segment, r) keeps its phase's NT taps in registers and walks UPP consecutive inputs p of
// its segment: per output one new sample from shared memory (the same address for all lanes of a segment), NT shifts of
// the sample window (register renaming: the walk is unrolled) and 2*NT multiply-adds -- against one sample load, one tap
// load and index arithmetic PER TAP in the kernel above.  Same sums in the same order (inputs ascending: k descending,
// starting from the carried partial sum); taps past the end of ir and inputs outside the push enter as exact zeros.
constexpr int UPP = 32;  // inputs a thread walks
template <typename T, int NT>
__global__ void __launch_bounds__(256) k_upsample_phase(const cx<T>* __restrict__ in, long long in_stride, long long len,
                                                        const cx<T>* __restrict__ acc_in, cx<T>* __restrict__ acc_out,
                                                        const T* __restrict__ ir, int L, int Q, int segs, long long j0, long long m0,
                                                        long long n_out, cx<T>* __restrict__ out, long long out_stride,
                                                        cx<T>* __restrict__ out2, long long out2_stride, long long out_split) {
    extern __shared__ __align__(16) unsigned char up_smem[];
    cx<T>* xs = reinterpret_cast<cx<T>*>(up_smem);  // inputs p_t0 - NT + 1 ... p_t0 + segs*UPP - 1
    const int s = blockIdx.y;
    const cx<T>* src = in + (long long)s * in_stride;
    const long long p_base = m0 / Q;  // input of the push's first output
    const long long p_t0 = p_base + (long long)blockIdx.x * (segs * UPP);
    const int n_x = segs * UPP + NT - 1;
    for (int i = threadIdx.x; i < n_x; i += blockDim.x) {
        const long long p = p_t0 - (NT - 1) + i;
        xs[i] = (p >= j0 && p < j0 + len) ? ld_cx(&src[p - j0]) : cx<T>((T)0, (T)0);
    }
    const int seg = threadIdx.x / Q, r = threadIdx.x - seg * Q;
    T h[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) h[k] = (seg < segs && r + k * Q < L) ? ir[r + k * Q] : (T)0;
    __syncthreads();
    if (seg >= segs) return;
    const int x0 = seg * UPP;  // xs index of input (first input of the segment) - (NT - 1)
    cx<T> w[NT];               // w[k] = x[p - k]
#pragma unroll
    for (int k = 1; k < NT; ++k) w[k] = xs[x0 + NT - 1 - k];
    const long long total = n_out + L;
    const long long o_first = (p_t0 + x0) * Q + r - m0, o_last = o_first + (long long)(UPP - 1) * Q;
    if (o_first >= L && o_last < n_out && (out2 == nullptr || o_last < out_split)) {
        // all of this thread's outputs are whole ones of the first destination: no carried sums, no bounds
        cx<T>* dst = out + (long long)s * out_stride + o_first;
#pragma unroll
        for (int i = 0; i < UPP; ++i) {
            w[0] = xs[x0 + NT - 1 + i];
            cx<T> acc((T)0, (T)0);
#pragma unroll
            for (int k = NT - 1; k >= 0; --k) {
                acc.x = fma(w[k].x, h[k], acc.x);
                acc.y = fma(w[k].y, h[k], acc.y);
            }
            st_cx(dst + (long long)i * Q, acc);
#pragma unroll
            for (int k = NT - 1; k >= 1; --k) w[k] = w[k - 1];
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < UPP; ++i) {
        w[0] = xs[x0 + NT - 1 + i];
        const long long q = (p_t0 + x0 + i) * Q + r;
        const long long o = q - m0;
        if (o >= 0 && o < total) {
            cx<T> acc = (o < L) ? ld_cx(&acc_in[(long long)s * L + o]) : cx<T>((T)0, (T)0);
#pragma unroll
            for (int k = NT - 1; k >= 0; --k) {
                acc.x = fma(w[k].x, h[k], acc.x);
                acc.y = fma(w[k].y, h[k], acc.y);
            }
            if (o < n_out) {
                if (out2 != nullptr && o >= out_split) st_cx(&out2[(long long)s * out2_stride + (o - out_split)], acc);
                else st_cx(&out[(long long)s * out_stride + o], acc);
            } else {
                st_cx(&acc_out[(long long)s * L + (o - n_out)], acc);
            }
        }
#pragma unroll
        for (int k = NT - 1; k >= 1; --k) w[k] = w[k - 1];
    }
}

template <typename T, int NT>
cudaError_t launch_upsample_phase(const void* in, long long in_stride, long long len, const void* acc_in, void* acc_out, const T* ir, int L,
                                  RateState rate, long long n_out, void* out, long long out_stride, int n_streams, cudaStream_t st, void* out2,
                                  long long out2_stride, long long out_split) {
    const int Q = (int)rate.Q, segs = 256 / Q;
    const long long p_base = rate.m0 / Q, p_last = (rate.m0 + n_out + L - 1) / Q;
    const long long tiles = (p_last - p_base) / (segs * UPP) + 1;
    const size_t smem = (size_t)(segs * UPP + NT - 1) * 2 * sizeof(T);
    dim3 grid((unsigned)tiles, (unsigned)n_streams);
    k_upsample_phase<T, NT><<<grid, segs * Q, smem, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len, reinterpret_cast<const cx<T>*>(acc_in),
                                                          reinterpret_cast<cx<T>*>(acc_out), ir, L, Q, segs, rate.j0, rate.m0, n_out,
                                                          reinterpret_cast<cx<T>*>(out), out_stride, reinterpret_cast<cx<T>*>(out2), out2_stride, out_split);
    return cudaGetLastError();
}

template <typename T> bool upsample_tiled_supported(RateState rate, int L) {
    if (!(rate.P == 1 && rate.Q >= 1 && rate.Q < (1LL << 30) && L <= 8192)) return false;
    const int x_cap = (int)(UP_TILE / rate.Q + L / rate.Q + 4);
    return (size_t)((L + 1) & ~1) * sizeof(T) + (size_t)x_cap * 2 * sizeof(T) <= 200 * 1024;
}

template <typename T>
cudaError_t launch_upsample(const void* in, long long in_stride, long long len, const void* acc_in, void* acc_out,
                            const T* ir, int L, RateState rate, long long n_out, void* out, long long out_stride,
                            int n_streams, cudaStream_t st, void* out2, long long out2_stride, long long out_split) {
    if (upsample_phase_supported(rate, L, n_out)) {
        // a phase per thread, its taps in registers (rates like 48 kS/s -> 2.4 MS/s: Q = 50, 11 taps per phase)
        const int nt = (int)((L + rate.Q - 1) / rate.Q);
        if (nt <= 4) return launch_upsample_phase<T, 4>(in, in_stride, len, acc_in, acc_out, ir, L, rate, n_out, out, out_stride, n_streams, st, out2, out2_stride, out_split);
        if (nt <= 8) return launch_upsample_phase<T, 8>(in, in_stride, len, acc_in, acc_out, ir, L, rate, n_out, out, out_stride, n_streams, st, out2, out2_stride, out_split);
        if (nt <= 12) return launch_upsample_phase<T, 12>(in, in_stride, len, acc_in, acc_out, ir, L, rate, n_out, out, out_stride, n_streams, st, out2, out2_stride, out_split);
        return launch_upsample_phase<T, 16>(in, in_stride, len, acc_in, acc_out, ir, L, rate, n_out, out, out_stride, n_streams, st, out2, out2_stride, out_split);
    }
    if (rate.P == 1 && rate.Q >= 1 && rate.Q < (1LL << 30) && L <= 8192) {
        // inputs per tile: at most UP_TILE / Q + L / Q + 2
        const int x_cap = (int)(UP_TILE / rate.Q + L / rate.Q + 4);
        const size_t smem = (size_t)((L + 1) & ~1) * sizeof(T) + (size_t)x_cap * 2 * sizeof(T);
        if (smem <= 200 * 1024) {
            const long long total = n_out + L;
            auto k = k_upsample_tiled<T>;
            cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            dim3 grid((unsigned)((total + UP_TILE - 1) / UP_TILE), (unsigned)n_streams);
            k<<<grid, 256, smem, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len, reinterpret_cast<const cx<T>*>(acc_in),
                                       reinterpret_cast<cx<T>*>(acc_out), ir, L, (int)rate.Q, rate.j0, rate.m0, n_out,
                                       reinterpret_cast<cx<T>*>(out), out_stride, x_cap, reinterpret_cast<cx<T>*>(out2), out2_stride, out_split);
            return cudaGetLastError();
        }
    }
    if (out2 != nullptr) return cudaErrorInvalidValue;  // the split destination is the tiled kernel's (callers check upsample_tiled_supported)
    const long long total = n_out + L;
    dim3 grid((unsigned)((total + 255) / 256), (unsigned)n_streams);
    k_upsample<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len,
                                        reinterpret_cast<const cx<T>*>(acc_in), reinterpret_cast<cx<T>*>(acc_out), ir,
                                        L, rate, n_out, reinterpret_cast<cx<T>*>(out), out_stride);
    return cudaGetLastError();
}

// The same with the input positions from tables (rates that are not integer valued): qpos[p] = output cell (relative
// to this push's first output) that input p starts at, cnt[i] = number of inputs with qpos <= i.
template <typename T>
__global__ void __launch_bounds__(256) k_upsample_idx(const cx<T>* __restrict__ in, long long in_stride, const cx<T>* __restrict__ acc_in,
                                                      cx<T>* __restrict__ acc_out, const T* __restrict__ ir, int L, const int* __restrict__ qpos,
                                                      const int* __restrict__ cnt, long long n_out, cx<T>* __restrict__ out, long long out_stride) {
    const int s = blockIdx.y;
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_out + L) return;
    const cx<T>* src = in + (long long)s * in_stride;
    cx<T> acc = (o < L) ? ld_cx(&acc_in[(long long)s * L + o]) : cx<T>((T)0, (T)0);
    const int p_hi = cnt[o] - 1;
    const int p_lo = (o - L >= 0) ? cnt[o - L] : 0;
    for (int p = p_lo; p <= p_hi; ++p) {  // input order, like the ring (resampling.rs:239-246)
        const int t = (int)(o - qpos[p]);
        if (t >= 0 && t < L) {
            const cx<T> x = ld_cx(&src[p]);
            const T h = ir[t];
            acc.x = fma(x.x, h, acc.x);
            acc.y = fma(x.y, h, acc.y);
        }
    }
    if (o < n_out) st_cx(&out[(long long)s * out_stride + o], acc);
    else st_cx(&acc_out[(long long)s * L + (o - n_out)], acc);
}
template <typename T>
cudaError_t launch_upsample_indexed(const void* in, long long in_stride, long long len, const void* acc_in, void* acc_out, const T* ir, int L,
                                    const int* qpos, const int* cnt, long long n_out, void* out, long long out_stride, int n_streams,
                                    cudaStream_t st) {
    (void)len;
    const long long total = n_out + L;
    dim3 grid((unsigned)((total + 255) / 256), (unsigned)n_streams);
    k_upsample_idx<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<const cx<T>*>(acc_in),
                                            reinterpret_cast<cx<T>*>(acc_out), ir, L, qpos, cnt, n_out, reinterpret_cast<cx<T>*>(out), out_stride);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// FmDemod, src/blocks/modulation.rs:116-126
// ---------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ T atan2_t(T y, T x);
template <> __device__ __forceinline__ float atan2_t<float>(float y, float x) { return atan2f(y, x); }
template <> __device__ __forceinline__ double atan2_t<double>(double y, double x) { return atan2(y, x); }

template <typename T>
__global__ void __launch_bounds__(256) k_fmdemod(const cx<T>* __restrict__ in, long long in_stride,
                                                 cx<T>* __restrict__ out, long long out_stride, long long len,
                                                 const cx<T>* __restrict__ prev_sample,
                                                 const cx<T>* __restrict__ last_output, int has_prev, T factor) {
    const int s = blockIdx.y;
    const cx<T>* src = in + (long long)s * in_stride;
    cx<T>* dst = out + (long long)s * out_stride;
    map_stream<T>(src, dst, len, [&](long long t, cx<T> v) {
        if (t == 0 && !has_prev) return ld_cx(&last_output[s]);  // repeat the previous output value (modulation.rs:119-124)
        const cx<T> prev = (t == 0) ? ld_cx(&prev_sample[s]) : ld_cx(&src[t - 1]);  // the neighbour's sample: an L1 hit
        const cx<T> p = cmulc(v, prev);
        return cx<T>(atan2_t<T>(p.y, p.x) * factor, (T)0);
    });
}
template <typename T>
__global__ void k_fm_state(const cx<T>* __restrict__ in, long long in_stride, const cx<T>* __restrict__ out,
                           long long out_stride, long long len, cx<T>* prev_sample, cx<T>* last_output, int n_streams) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n_streams) {
        st_cx(&prev_sample[s], ld_cx(&in[(long long)s * in_stride + len - 1]));
        st_cx(&last_output[s], ld_cx(&out[(long long)s * out_stride + len - 1]));
    }
}
template <typename T>
cudaError_t launch_fmdemod(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                           int n_streams, void* prev_sample, void* last_output, int has_prev, double factor,
                           cudaStream_t st) {
    if (len <= 0) return cudaSuccess;
    dim3 grid(map_grid_x(len, n_streams), (unsigned)n_streams);
    k_fmdemod<T><<<grid, 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<cx<T>*>(out),
                                       out_stride, len, reinterpret_cast<const cx<T>*>(prev_sample),
                                       reinterpret_cast<const cx<T>*>(last_output), has_prev, (T)factor);
    k_fm_state<T><<<(n_streams + 127) / 128, 128, 0, st>>>(
        reinterpret_cast<const cx<T>*>(in), in_stride, reinterpret_cast<const cx<T>*>(out), out_stride, len,
        reinterpret_cast<cx<T>*>(prev_sample), reinterpret_cast<cx<T>*>(last_output), n_streams);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// metering::level (src/metering.rs:21-30): mean square norm of a chunk, accumulated in f64.
// One CTA per (chunk, stream); the f64 partial sums are combined in a fixed order (deterministic).
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_level(const cx<T>* __restrict__ in, long long in_stride, long long chunk_len,
                                               double* __restrict__ out, long long n_chunks) {
    __shared__ double part[8];
    const cx<T>* src = in + (long long)blockIdx.y * in_stride + (long long)blockIdx.x * chunk_len;
    double acc = 0.0;
    for (long long t = threadIdx.x; t < chunk_len; t += blockDim.x) {
        const cx<T> v = ld_cx(&src[t]);
        const T nsq = v.x * v.x + v.y * v.y;  // norm_sqr in Flt, then to_f64 (metering.rs:27)
        acc += (double)nsq;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0;
        for (int w = 0; w < 8; ++w) sum += part[w];
        out[(long long)blockIdx.y * n_chunks + blockIdx.x] = sum / (double)chunk_len;
    }
}
template <typename T>
cudaError_t launch_level(const void* in, long long in_stride, long long chunk_len, long long n_chunks, int n_streams, double* out,
                         cudaStream_t st) {
    if (n_chunks <= 0 || chunk_len <= 0) return cudaSuccess;
    k_level<T><<<dim3((unsigned)n_chunks, (unsigned)n_streams), 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, chunk_len, out,
                                                                             n_chunks);
    return cudaGetLastError();
}

#define RR_INST(T)                                                                                                     \
    template cudaError_t launch_freqshift<T>(const void*, long long, void*, long long, long long, int,                 \
                                             const NcoStream*, long long, cudaStream_t);                                                          \
    template cudaError_t launch_gain<T>(const void*, long long, void*, long long, long long, int, double,              \
                                        cudaStream_t);                                                                 \
    template cudaError_t launch_copy2d<T>(const void*, long long, void*, long long, long long, int, cudaStream_t);     \
    template cudaError_t launch_downsample<T>(const void*, long long, long long, const void*, void*, const T*, int,    \
                                              RateState, long long, void*, long long, int, cudaStream_t);              \
    template cudaError_t launch_upsample<T>(const void*, long long, long long, const void*, void*, const T*, int,      \
                                            RateState, long long, void*, long long, int, cudaStream_t, void*, long long, long long); \
    template bool upsample_tiled_supported<T>(RateState, int);                                                         \
    template cudaError_t launch_downsample_indexed<T>(const void*, long long, long long, const void*, void*, const T*, int, const int*, \
                                                      long long, void*, long long, int, cudaStream_t);                 \
    template cudaError_t launch_upsample_indexed<T>(const void*, long long, long long, const void*, void*, const T*, int, const int*,   \
                                                    const int*, long long, void*, long long, int, cudaStream_t);       \
    template cudaError_t launch_fmdemod<T>(const void*, long long, void*, long long, long long, int, void*, void*,     \
                                           int, double, cudaStream_t);                                                 \
    template cudaError_t launch_level<T>(const void*, long long, long long, long long, int, double*, cudaStream_t);
RR_INST(float)
RR_INST(double)
#undef RR_INST

}  // namespace rr
