// Summed-output pushes: every stream's output of a push added into one row (rr_chain_push_summed[_device]).
//
// The row is out[t] = sum over s ascending of y_s[t], y_s[t] the T-rounded output a per-stream push writes for stream
// s, accumulated in f64 from +0.0 and rounded once to T.  Every output sample is owned by one thread, which walks the
// streams in order: no atomics, no partial sums split over streams, so the row does not depend on the grid.
//
//   k_synth       Upsampler (integer factor, k_upsample_phase's form) -> FreqShifter as the chain's last two stages:
//                 interpolation, mixing and the sum in one kernel.  Reads the S inputs at the low rate and writes one
//                 row; the S full-rate rows of a per-stream push are never formed.
//   k_stream_sum  every other chain: the per-stream rows (in scratch) added into the row.
// sm_100a.
#include "rr_chain_os.cuh"

namespace rr {

// k_freqshift's mixing of one sample, with the products it contracts (rr_stage_kernels.cu, nco_phasor then cmul)
// written as the fma's its SASS holds: the same roundings in both kernels.
template <typename T> __device__ __forceinline__ cx<T> mix_like_freqshift(cx<T> v, uint32_t i, uint32_t denom, int sign, T start) {
    const T tau = (T)6.283185307179586476925286766559;
    const T frac = (T)i / (T)denom;
    const T ph = fma(frac, sign < 0 ? -tau : tau, start);
    T s, c;
    sincos_t<T>(ph, &s, &c);
    return cx<T>(fma(v.x, c, -(v.y * s)), fma(v.x, s, v.y * c));
}

// asynchronous 8/16-byte copy of one complex sample into shared memory; a zero fill where !valid (nothing is read)
template <typename T> __device__ __forceinline__ void cp_async_cx(cx<T>* dst, const cx<T>* src, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;\n" ::"r"(d), "l"(src), "n"((int)(2 * sizeof(T))),
                 "r"(valid ? (int)(2 * sizeof(T)) : 0));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_prev() { asm volatile("cp.async.wait_group 1;\n" ::); }

// Grid: pend_blocks CTAs for the row samples t < pending (read from the Upsampler's staging buffer), then one CTA per
// tile of segs*UPPS inputs.  Tile thread (seg, r) owns the UPPS outputs q = p*Q + r of inputs p = p_t0 + seg*UPPS + i:
// for each stream it computes them exactly as k_upsample_phase does (taps in registers, the same fma chain from the
// carried partial sum), mixes the row's part as k_freqshift does and adds it into its f64 accumulators.  Outputs behind
// the row go, pre-NCO, where a per-stream push leaves them: the Upsampler's next pending part and carried sums.  The
// window of stream s+1 is copied into shared memory (cp.async, double-buffered) while stream s is computed.
template <typename T, int NT, int UPPS>
__global__ void __launch_bounds__(256) k_synth(const SynthArgs a, int n_streams, int segs, int pend_blocks) {
    extern __shared__ __align__(16) unsigned char synth_smem[];
    const cx<T>* in = reinterpret_cast<const cx<T>*>(a.in);
    const cx<T>* pend = reinterpret_cast<const cx<T>*>(a.pend);
    cx<T>* out = reinterpret_cast<cx<T>*>(a.out);
    double ax[UPPS], ay[UPPS];
#pragma unroll
    for (int i = 0; i < UPPS; ++i) ax[i] = ay[i] = 0.0;

    if ((int)blockIdx.x < pend_blocks) {
        const long long t0 = (long long)blockIdx.x * blockDim.x * UPPS + threadIdx.x;
        for (int s = 0; s < n_streams; ++s) {
            const NcoStream ns = a.nco[s];
            cx<T> v[UPPS];
#pragma unroll
            for (int i = 0; i < UPPS; ++i) {
                const long long t = t0 + (long long)i * blockDim.x;
                if (t < a.pending) v[i] = ld_cx(&pend[(long long)s * a.obuf_stride + t]);
            }
#pragma unroll
            for (int i = 0; i < UPPS; ++i) {
                const long long t = t0 + (long long)i * blockDim.x;
                if (t < a.pending) {
                    const uint32_t k = (uint32_t)(((unsigned long long)ns.idx + (unsigned long long)t) % ns.denom);
                    const cx<T> m = mix_like_freqshift<T>(v[i], mulmod_u32(ns.numer_abs, k, ns.denom), ns.denom, ns.sign, (T)ns.start_phase);
                    ax[i] += (double)m.x;
                    ay[i] += (double)m.y;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < UPPS; ++i) {
            const long long t = t0 + (long long)i * blockDim.x;
            if (t < a.pending) st_cx(&out[t], cx<T>((T)ax[i], (T)ay[i]));
        }
        return;
    }

    const int Q = a.Q, L = a.L;
    const int n_x = segs * UPPS + NT - 1;
    const int x_pitch = (n_x + 1) & ~1;
    cx<T>* xbuf = reinterpret_cast<cx<T>*>(synth_smem);  // [2][x_pitch]: inputs p_t0 - NT + 1 ... p_t0 + segs*UPPS - 1
    const long long p_t0 = a.m0 / Q + (long long)(blockIdx.x - pend_blocks) * (segs * UPPS);
    auto stage = [&](int s, int buf) {
        const cx<T>* src = in + (long long)s * a.in_stride;
        for (int i = threadIdx.x; i < n_x; i += blockDim.x) {
            const long long p = p_t0 - (NT - 1) + i;
            const bool ok = p >= a.j0 && p < a.j0 + a.len;
            cp_async_cx<T>(&xbuf[buf * x_pitch + i], ok ? &src[p - a.j0] : in, ok);
        }
        cp_async_commit();
    };

    const int seg = threadIdx.x / Q, r = threadIdx.x - seg * Q;
    const bool active = seg < segs;
    T h[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) h[k] = (active && r + k * Q < L) ? reinterpret_cast<const T*>(a.ir)[r + k * Q] : (T)0;
    const int x0 = seg * UPPS;
    const long long total = a.n_new + L;
    const long long o_first = (p_t0 + x0) * Q + r - a.m0;  // output index of i = 0 (relative to m0; may be < 0)
    const cx<T>* acc_in = reinterpret_cast<const cx<T>*>(a.acc_in);
    cx<T>* acc_out = reinterpret_cast<cx<T>*>(a.acc_out);
    cx<T>* rem = reinterpret_cast<cx<T>*>(a.rem);

    stage(0, 0);
    for (int s = 0; s < n_streams; ++s) {
        if (s + 1 < n_streams) stage(s + 1, (s + 1) & 1);
        else cp_async_commit();  // an empty group: the wait below always leaves exactly the newest one in flight
        cp_async_wait_prev();
        __syncthreads();
        if (active) {
            const cx<T>* xs = xbuf + (s & 1) * x_pitch;
            const NcoStream ns = a.nco[s];
            const T start = (T)ns.start_phase;
            // NCO table position of output i: (idx + pending + o) mod denom; i_k = numer*k mod denom advances by a fixed
            // step per output of this thread (Q samples apart) -- the same integers k_freqshift derives per sample
            long long k0 = ((long long)ns.idx + a.pending + o_first) % (long long)ns.denom;
            if (k0 < 0) k0 += ns.denom;
            uint32_t ik = mulmod_u32(ns.numer_abs, (uint32_t)k0, ns.denom);
            const uint32_t step = mulmod_u32(ns.numer_abs, (uint32_t)Q % ns.denom, ns.denom);
            cx<T> w[NT];  // w[k] = x[p - k]
#pragma unroll
            for (int k = 1; k < NT; ++k) w[k] = xs[x0 + NT - 1 - k];
#pragma unroll
            for (int i = 0; i < UPPS; ++i) {
                w[0] = xs[x0 + NT - 1 + i];
                const long long o = o_first + (long long)i * Q;
                if (o >= 0 && o < total) {
                    cx<T> y = (o < L) ? ld_cx(&acc_in[(long long)s * L + o]) : cx<T>((T)0, (T)0);
#pragma unroll
                    for (int k = NT - 1; k >= 0; --k) {
                        y.x = fma(w[k].x, h[k], y.x);
                        y.y = fma(w[k].y, h[k], y.y);
                    }
                    if (o < a.split) {
                        const cx<T> m = mix_like_freqshift<T>(y, ik, ns.denom, ns.sign, start);
                        ax[i] += (double)m.x;
                        ay[i] += (double)m.y;
                    } else if (o < a.n_new) {
                        st_cx(&rem[(long long)s * a.obuf_stride + (o - a.split)], y);
                    } else {
                        st_cx(&acc_out[(long long)s * L + (o - a.n_new)], y);
                    }
                }
                ik = addmod_u32(ik, step, ns.denom);
#pragma unroll
                for (int k = NT - 1; k >= 1; --k) w[k] = w[k - 1];
            }
        }
        __syncthreads();  // buffer (s & 1) is refilled for stream s + 2 next
    }
    if (!active) return;
#pragma unroll
    for (int i = 0; i < UPPS; ++i) {
        const long long o = o_first + (long long)i * Q;
        if (o >= 0 && o < a.split) st_cx(&out[a.pending + o], cx<T>((T)ax[i], (T)ay[i]));
    }
}

template <typename T, int NT, int UPPS>
cudaError_t launch_synth_nt(const SynthArgs& a, int n_streams, cudaStream_t st) {
    const int segs = 256 / a.Q;
    const int threads = segs * a.Q;
    const long long p_base = a.m0 / a.Q, p_last = (a.m0 + a.n_new + a.L - 1) / a.Q;
    const long long tiles = (p_last - p_base) / (segs * UPPS) + 1;
    const long long pend_blocks = (a.pending + (long long)threads * UPPS - 1) / ((long long)threads * UPPS);
    const size_t smem = 2 * (size_t)((segs * UPPS + NT - 1 + 1) & ~1) * 2 * sizeof(T);
    if (pend_blocks + tiles >= (1LL << 31)) return cudaErrorInvalidValue;
    k_synth<T, NT, UPPS><<<(unsigned)(pend_blocks + tiles), threads, smem, st>>>(a, n_streams, segs, (int)pend_blocks);
    return cudaGetLastError();
}

template <typename T, int UPPS> cudaError_t launch_synth_upps(const SynthArgs& a, int n_streams, cudaStream_t st) {
    const int nt = (a.L + a.Q - 1) / a.Q;
    if (nt <= 4) return launch_synth_nt<T, 4, UPPS>(a, n_streams, st);
    if (nt <= 8) return launch_synth_nt<T, 8, UPPS>(a, n_streams, st);
    if (nt <= 12) return launch_synth_nt<T, 12, UPPS>(a, n_streams, st);
    return launch_synth_nt<T, 16, UPPS>(a, n_streams, st);
}

template <typename T> cudaError_t launch_synth(const SynthArgs& a, int n_streams, int sm_count, cudaStream_t st) {
    RateState rate{1, a.Q, a.j0, a.m0};
    if (!upsample_phase_supported(rate, a.L, a.n_new) || a.split < 0 || a.split > a.n_new || a.pending < 0) return cudaErrorInvalidValue;
    // a CTA walks every stream of its tile: eight outputs per thread when that still gives every SM two CTAs, two
    // otherwise (short pushes)
    const int segs = 256 / a.Q;
    const long long tiles8 = ((a.m0 + a.n_new + a.L - 1) / a.Q - a.m0 / a.Q) / (segs * 8) + 1;
    if (tiles8 >= 2LL * sm_count) return launch_synth_upps<T, 8>(a, n_streams, st);
    return launch_synth_upps<T, 2>(a, n_streams, st);
}

// One thread per row sample; kStreamsInFlight loads of consecutive streams are issued before they are added, in order.
constexpr int kStreamsInFlight = 8;
template <typename T>
__global__ void __launch_bounds__(256) k_stream_sum(const cx<T>* __restrict__ in, long long in_stride, long long len, int n_streams,
                                                    cx<T>* __restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= len) return;
    double ax = 0.0, ay = 0.0;
    int s = 0;
    for (; s + kStreamsInFlight <= n_streams; s += kStreamsInFlight) {
        cx<T> v[kStreamsInFlight];
#pragma unroll
        for (int u = 0; u < kStreamsInFlight; ++u) v[u] = ld_cx(&in[(long long)(s + u) * in_stride + t]);
#pragma unroll
        for (int u = 0; u < kStreamsInFlight; ++u) {
            ax += (double)v[u].x;
            ay += (double)v[u].y;
        }
    }
    for (; s < n_streams; ++s) {
        const cx<T> v = ld_cx(&in[(long long)s * in_stride + t]);
        ax += (double)v.x;
        ay += (double)v.y;
    }
    st_cx(&out[t], cx<T>((T)ax, (T)ay));
}

template <typename T>
cudaError_t launch_stream_sum(const void* in, long long in_stride, long long len, int n_streams, void* out, cudaStream_t st) {
    if (len <= 0) return cudaSuccess;
    k_stream_sum<T><<<(unsigned)((len + 255) / 256), 256, 0, st>>>(reinterpret_cast<const cx<T>*>(in), in_stride, len, n_streams,
                                                                  reinterpret_cast<cx<T>*>(out));
    return cudaGetLastError();
}

template cudaError_t launch_synth<float>(const SynthArgs&, int, int, cudaStream_t);
template cudaError_t launch_synth<double>(const SynthArgs&, int, int, cudaStream_t);
template cudaError_t launch_stream_sum<float>(const void*, long long, long long, int, void*, cudaStream_t);
template cudaError_t launch_stream_sum<double>(const void*, long long, long long, int, void*, cudaStream_t);

}  // namespace rr
