// Host side of the C ABI (include/radiorust_b200.h): contexts, pinned pool,
// design-math exports and the chain object that sequences the sm_100a kernels.
//
// A chain replays, for `n_streams` streams in lock step, what the reference's
// per-block Tokio tasks do for one stream (SURVEY.md 3.2): every
// rr_chain_push is "n_chunks Signal::Samples messages per stream", every
// rr_chain_event is one in-band Signal::Event.  All per-block bookkeeping that
// the reference keeps in task locals (Filter's has-history flag
// filters.rs:164, Downsampler's pos/ring resampling.rs:65-67, FreqShifter's
// phase_idx transform.rs:308, FmDemod's previous sample modulation.rs:103) is
// host scalars here plus device-resident sample state; the sample arithmetic
// itself only ever runs in the CUDA kernels -- there is no CPU fallback.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <complex>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/radiorust_b200.h"
#include "rr_design.h"
#include "rr_kernels.h"

namespace {

thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
int fail_cuda(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return RR_ERR_CUDA;
}
#define RR_CUDA(expr)                                     \
    do {                                                  \
        cudaError_t e__ = (expr);                         \
        if (e__ != cudaSuccess) return fail_cuda(e__, #expr); \
    } while (0)
#define RR_TRY(expr)              \
    do {                          \
        int r__ = (expr);         \
        if (r__ != RR_OK) return r__; \
    } while (0)
// kernel launch wrapper: counts launches (rr_kernel_launch_count)
#define RR_LAUNCH(n_kernels, expr)                        \
    do {                                                  \
        cudaError_t e__ = (expr);                         \
        if (e__ != cudaSuccess) return fail_cuda(e__, #expr); \
        g_launches.fetch_add((n_kernels));                \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    // grow-only; contents are NOT preserved
    // zero = true clears a NEW allocation on `st` (the stream whose kernels use the buffer: a memset on the legacy
    // stream would not be ordered against a non-blocking stream)
    int ensure(size_t need, bool zero = false, cudaStream_t st = nullptr) {
        if (need <= bytes && p) {
            return RR_OK;
        }
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        if (need == 0) need = 16;
        cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess) {
            p = nullptr;
            g_err = std::string("cudaMalloc: ") + cudaGetErrorString(e);
            return e == cudaErrorMemoryAllocation ? RR_ERR_NOMEM : RR_ERR_CUDA;
        }
        bytes = need;
        if (zero) {
            e = cudaMemsetAsync(p, 0, need, st);
            if (e != cudaSuccess) return fail_cuda(e, "cudaMemsetAsync");
        }
        return RR_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};

struct Shape {
    size_t chunk_len = 0, n_chunks = 0;
    double rate = 0.0;
    size_t len() const { return chunk_len * n_chunks; }
};

struct View {
    const void* p = nullptr;
    long long stride = 0;
    Shape sh;
};

// ---- host mirror of one stream's NCO (transform.rs:307-309) -----------------
struct NcoHost {
    int64_t numer = 0, denom = 1;
    uint64_t idx = 0;
    double start_phase = 0.0;  // value representable in Flt
    bool has_table = false;    // phase_vec non-empty
};

// small, copyable host state per stage: everything needed to know the output
// shape of a push without touching the device (dry run == real run)
struct StageHost {
    // FILTER
    double f_sr = NAN;
    size_t f_n = 0;
    int f_seg = 0;  // chunks received in the current segment (since start / redesign / interrupt), saturates at 2
    bool f_dirty = true;
    // RESAMPLERS
    double r_in_rate = NAN;
    bool r_valid = false;
    int r_L = 0;
    long long P = 1, Q = 1, j0 = 0, m0 = 0;
    size_t r_pending = 0;
    // rates that are not integer valued: the firing pattern follows the reference's f64 `pos` recurrence
    // (resampling.rs:67,109-111 / :197,247-266) step by step instead of the exact rational form
    bool r_indexed = false;
    double r_pos = 0.0;
    // FMDEMOD
    bool fm_has_prev = false;
    // FREQSHIFT
    double n_sr = NAN;
    // RECHUNK: samples of the partial chunk and their sample rate
    size_t rc_pending = 0;
    double rc_rate = NAN;
    // OVERLAP: chunks kept (< chunk_count), their length and sample rate
    size_t ov_hist = 0, ov_len = 0;
    double ov_rate = NAN;
};

struct StageAct {
    bool active = false;       // the stage received samples in this push
    bool redesign = false;     // filter response / resampler taps must be rebuilt
    bool first_is_history = false;
    size_t n_new = 0;          // resampler: samples produced by this push
    size_t pending_before = 0;
    long long j0 = 0, m0 = 0;  // resampler counters before the push
    double pos0 = 0.0;         // indexed resampler: `pos` before the push
    bool nco_recalc = false;
    int seg_before = 0;        // filter: chunks of the current segment seen before this push
    bool lost = false;         // Rechunker: the partial chunk was dropped (SamplesLost goes downstream first)
    Shape out;
};

inline long long floordiv128(long long a, long long b, long long c) { return (long long)(((__int128)a * b) / c); }
inline long long ceildiv128(long long a, long long b, long long c) { return (long long)(((__int128)a * b + (c - 1)) / c); }

bool integer_valued(double x) { return std::isfinite(x) && x >= 0.0 && x < 9.0e15 && std::floor(x) == x; }

}  // namespace

struct rr_ctx {
    int device = 0;
    int sm_count = 0;
};


// Recycling pool of pinned host buffers (the chain-edge stand-in for bufferpool.rs:187-222).  `idle` is the
// recycler channel (FIFO, bufferpool.rs:82-90 sends, :203-207 / :213-219 receive); `live` are the buffers handed out.
struct rr_pool {
    rr_ctx* ctx = nullptr;
    std::mutex mu;
    struct Buf {
        void* p;
        size_t cap;
    };
    std::deque<Buf> idle;
    std::unordered_map<void*, size_t> live;
    uint64_t n_alloc = 0, n_reuse = 0;
};

namespace {

struct Stage {
    rr_stage_desc d{};
    StageHost h;
    // FREQSHIFT
    std::vector<double> shift;
    std::vector<uint8_t> shift_dirty;
    bool any_shift_dirty = true;
    std::vector<NcoHost> nco_h;
    std::vector<rr::NcoStream> nco_stage;  // upload staging
    DevBuf nco_d;
    // FILTER
    DevBuf hperm, tw;
    DevBuf hist2[2];  // [S][2n] post-NCO samples preceding the next push (older chunk | newer chunk), ping-pong
    int hist_cur = 0;
    // >= 0: this push's k_front already wrote entries [hist_fused_jfirst, hist_fused_jlo) of the new hist2
    long long hist_fused_jlo = -1, hist_fused_jfirst = 0;
    DevBuf ztmp;      // filter-output scratch of the unfused stateful path
    // chunk lengths that are not a power of two run on the kernels of the next power of two f_np (taps zero padded):
    // [history chunk | pushed chunks] is staged contiguously, transformed in chunks of f_np, and the wanted slice copied out
    size_t f_np = 0;
    DevBuf stg_in, stg_out, zero_chunk;
    // indexed resamplers: firing / position tables of the current push
    DevBuf idx_a, idx_b;
    std::vector<std::complex<double>> taps;  // windowed impulse response (Flt-rounded), for the polyphase tables
    bool taps_valid = false;
    // big overlap-save tables
    DevBuf big_h, big_twA, big_twB, big_twC, big_scratch;
    // RESAMPLERS
    DevBuf ir, tail[2], obuf[2];
    int tail_cur = 0, obuf_cur = 0;
    std::vector<double> ir_host_flt;  // taps as rounded to Flt
    bool ztail_stale = false;  // the polyphase path ran: tail[] must be rebuilt from the filter's hist2 before reuse
    // polyphase tables of the fused Filter -> Downsampler path (rebuilt when either block is redesigned)
    DevBuf gtab, twK;
    bool poly_valid = false, poly_tried = false;
    int poly_K = 0, poly_G = 0, poly_Lmax = 0, poly_V = 0;
    // k_poly2 (f32, Q == 1): its own table layout, K = 512
    DevBuf gtab2, twK2;
    bool poly2_tw_own = false;
    // rank-reduced front end (k_front) + k_poly2 on its output: coefficient table, low-rate table, scratch
    DevBuf acoef, gtab3, ubuf[2];
    long long ubuf_stride[2] = {-1, -1};  // layout the zeroed pad rows of each ubuf belong to
    // the last Lmax rows of u written by the previous push (in ubuf[ubuf_cur ^ 1]) are the history rows of the next
    // one as long as every push in between went through the front end
    int ubuf_cur = 0;
    bool ucache_valid = false;
    long long ucache_rows = 0;  // rows of the previous push
    // where the last Lmax rows of u of the previous front-end push live (either path leaves them behind)
    const void* ucache_ptr = nullptr;
    long long ucache_stride = 0;
    // k_fused (front end + low-rate part in one kernel): its kept rows (ping-pong) and its constant-memory slot
    DevBuf ukeep[2];
    int ukeep_cur = 0;
    int fused_slot = -1;
    bool fused_valid = false;
    bool front_valid = false;
    int front_rank = 0;
    double front_discarded = 0.0;
    // in/out = P/Q with Q > 1 (f32): front end of kFrontQRank columns shared by the Q phases, then k_poly on u
    bool frontq_valid = false;
    bool frontq_wide = false;  // k_front_wide (any P) instead of k_front (even P <= 254)
    int frontq_cols = 0;       // columns of u: 16 or 32
    int frontq_rank = 0;
    double frontq_discarded = 0.0;
    DevBuf acoef_q, gtab_q;
    bool poly2_valid = false;
    int poly2_G = 0, poly2_V = 0;
    size_t obuf_cap = 0;  // samples per stream in obuf
    std::vector<double> ir_host;
    // FMDEMOD
    DevBuf fm_prev, fm_last;
    // FMMOD: the phase accumulator per stream (Flt).  RECHUNK keeps its partial chunk in obuf[], OVERLAP its
    // history chunks in tail[] (both ping-pong)
    DevBuf fm_phase;
    size_t tail_cap = 0;  // OVERLAP: samples per stream in tail[]
    // FOURIER: window values (Flt) and twiddles of the current chunk length
    DevBuf fwin, ftw;
    size_t fwin_n = 0;
    // generic output buffer
    DevBuf out;
    size_t out_cap = 0;
};

}  // namespace

struct rr_chain {
    rr_ctx* ctx = nullptr;
    int dtype = RR_C32;
    size_t esz = 8;  // bytes per complex sample
    int S = 1;
    std::vector<Stage> st;
    cudaStream_t stream = nullptr;
    // rr_chain_push: two staging slots and two copy streams, so that the H2D copy of push k+1 runs while push k's
    // kernels and D2H copy are still in flight (PCIe is full duplex; the chain edges are the only PCIe traffic)
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    DevBuf stage_in[2], stage_out[2];
    DevBuf sum_rows;  // summed pushes off the k_synth route: the per-stream outputs, added into the caller's row
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    cudaEvent_t ev_copy = nullptr;
    int slot = 0;
    std::string plan;
    uint64_t samples_lost = 0;  // SamplesLost events generated by Rechunker / Overlapper stages
    bool push_mutated = false;  // the running push has passed its dry run and changed stage state
    bool allow_poly = true;  // rr_chain_set_fast_path
    bool allow_poly2 = true; // RR_DISABLE_POLY2=1: keep the generic polyphase kernel (k_poly) for f32 too
    size_t big_os_scratch_bytes = (size_t)2 << 30;  // RR_BIG_OS_SCRATCH_MB
    bool allow_sab = true;    // RR_DISABLE_SAB=1: short pushes keep one low-rate block (and inverse round) per stream
    bool allow_ucache = true; // RR_DISABLE_UCACHE=1: recompute the history rows of u from hist2 in every push
    bool allow_front = true; // RR_DISABLE_FRONT=1: k_poly2 on all P branches instead of the rank-reduced front end
    bool allow_fused = true; // RR_DISABLE_FUSED=1: k_front + k_poly2 (u through HBM) instead of k_fused
    int fused_min_streams = -1;  // streams from which k_fused is used (default: two per SM; RR_FUSED_MIN_STREAMS)
    long long fused_min_rows = 1;  // new rows (outputs) per stream and push from which k_fused is used (RR_FUSED_MIN_ROWS)
    // optional CUDA-event timing of the dominant kernel of a push (bench.py's roofline)
    bool timing = false;
    std::vector<cudaEvent_t> evs;  // pairs (start, stop), one per timed launch since rr_chain_set_timing
    size_t ev_used = 0;
    std::vector<std::string> ev_names;  // kernel name per pair
    std::string timed_kernel, breakdown;
    int timing_begin() {
        if (!timing) return 0;
        if (ev_used + 2 > evs.size()) {
            cudaEvent_t a = nullptr, b = nullptr;
            if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return 0;
            evs.push_back(a);
            evs.push_back(b);
        }
        cudaEventRecord(evs[ev_used], stream);
        return 1;
    }
    void timing_end(const char* name) {
        cudaEventRecord(evs[ev_used + 1], stream);
        ev_used += 2;
        if (ev_names.size() < ev_used / 2) ev_names.resize(ev_used / 2);
        ev_names[ev_used / 2 - 1] = name;
    }
};

namespace {
void chain_restart(rr_chain* c);
}

#define RR_TIMED_LAUNCH(c, name, n_kernels, expr)                        \
    do {                                                                 \
        const int t__ = (c)->timing_begin();                             \
        RR_LAUNCH(n_kernels, expr);                                      \
        if (t__) (c)->timing_end(name);                                  \
    } while (0)

namespace {

// ---------------------------------------------------------------------------
// shape logic shared by the dry run (capacity check, rr_chain_max_output) and
// the real run
// ---------------------------------------------------------------------------
int advance_stage(const rr_stage_desc& d, StageHost& h, const Shape& in, StageAct* act) {
    StageAct a;
    a.out = in;
    if (in.n_chunks == 0 || in.chunk_len == 0) {
        a.out.n_chunks = 0;
        *act = a;
        return RR_OK;
    }
    a.active = true;
    switch (d.kind) {
        case RR_STAGE_FREQSHIFT:
            a.nco_recalc = !(h.n_sr == in.rate);
            h.n_sr = in.rate;
            break;
        case RR_STAGE_GAIN:
        case RR_STAGE_FOURIER:
        case RR_STAGE_FMMOD:
            break;
        case RR_STAGE_RECHUNK: {
            // chunks.rs:71-79: a partial chunk of another sample rate is dropped and reported
            if (h.rc_pending > 0 && !(h.rc_rate == in.rate)) {
                h.rc_pending = 0;
                a.lost = true;
            }
            h.rc_rate = in.rate;
            const size_t ocl = (size_t)d.output_chunk_len;
            a.pending_before = h.rc_pending;
            a.n_new = in.len();
            const size_t total = h.rc_pending + a.n_new;
            a.out.chunk_len = ocl;
            a.out.n_chunks = total / ocl;
            h.rc_pending = total - a.out.n_chunks * ocl;
            break;
        }
        case RR_STAGE_OVERLAP: {
            const size_t k = (size_t)d.chunk_count;
            if (h.ov_hist > 0 && (h.ov_len != in.chunk_len || !(h.ov_rate == in.rate)))
                return fail(RR_ERR_UNSUPPORTED, "Overlapper: the chunks of one history must share length and sample rate");
            a.pending_before = h.ov_hist;
            const size_t tot = h.ov_hist + in.n_chunks;
            a.out.chunk_len = k * in.chunk_len;
            a.out.n_chunks = tot >= k ? tot - (k - 1) : 0;
            // chunks.rs:207-214: the length-weighted mean of the k sample rates, evaluated the same way
            double acc = 0.0;
            for (size_t i = 0; i < k; ++i) acc += in.rate * (double)in.chunk_len;
            a.out.rate = acc / (double)(k * in.chunk_len);
            h.ov_hist = std::min(k - 1, tot);
            h.ov_len = in.chunk_len;
            h.ov_rate = in.rate;
            break;
        }
        case RR_STAGE_FMDEMOD:
            a.first_is_history = !h.fm_has_prev;
            h.fm_has_prev = true;
            break;
        case RR_STAGE_FILTER: {
            // filters.rs:179-187: redesign on new params / sample rate / chunk length, and drop history
            a.redesign = h.f_dirty || !(h.f_sr == in.rate) || h.f_n != in.chunk_len;
            if (a.redesign) {
                h.f_dirty = false;
                h.f_sr = in.rate;
                h.f_n = in.chunk_len;
                h.f_seg = 0;
            }
            a.seg_before = h.f_seg;
            a.first_is_history = (h.f_seg == 0);  // filters.rs:240,260
            a.out.n_chunks = in.n_chunks - (a.first_is_history ? 1 : 0);
            h.f_seg = (int)std::min<size_t>(2, (size_t)h.f_seg + in.n_chunks);
            break;
        }
        case RR_STAGE_DOWNSAMPLE:
        case RR_STAGE_UPSAMPLE: {
            const bool down = d.kind == RR_STAGE_DOWNSAMPLE;
            if (!h.r_valid || !(h.r_in_rate == in.rate)) {  // resampling.rs:75 / :205
                const double in_rate = in.rate, out_rate = d.output_rate;
                if (!(in_rate >= 0.0)) return fail(RR_ERR_INVALID, "input sample rate must be positive");
                if (down && !(in_rate >= out_rate))
                    return fail(RR_ERR_INVALID, "input sample rate must be greater than or equal to output sample rate");
                if (!down && !(in_rate <= out_rate))
                    return fail(RR_ERR_INVALID, "input sample rate must be smaller than or equal to output sample rate");
                if (!down && !(d.bandwidth < in_rate))
                    return fail(RR_ERR_INVALID, "bandwidth must be smaller than input sample rate");
                const double margin = down ? (out_rate - d.bandwidth) / 2.0 : (in_rate - d.bandwidth) / 2.0;
                const double lf = std::ceil((down ? in_rate : out_rate) / margin * d.quality);
                if (!(lf > 0.0) || lf > 1.0e8) return fail(RR_ERR_INVALID, "resampler impulse response length out of range");
                if (in_rate == 0.0 || out_rate == 0.0) return fail(RR_ERR_INVALID, "resampler sample rates must be non-zero");
                h.r_indexed = !integer_valued(in_rate) || !integer_valued(out_rate);
                h.r_pos = 0.0;
                if (!h.r_indexed) {
                    long long Pn = (long long)in_rate, Qn = (long long)out_rate;
                    const long long g = std::gcd(Pn, Qn);
                    h.P = Pn / g;
                    h.Q = Qn / g;
                } else {
                    h.P = h.Q = 1;
                }
                h.j0 = 0;
                h.m0 = 0;
                h.r_L = (int)lf;
                h.r_in_rate = in_rate;
                h.r_valid = true;
                a.redesign = true;
            }
            const long long len = (long long)in.len();
            a.j0 = h.j0;
            a.m0 = h.m0;
            a.pos0 = h.r_pos;
            if (h.r_indexed) {
                // the reference's recurrence, literally (f64 `pos`): count the outputs of this push
                const double in_rate = in.rate, out_rate = d.output_rate;
                double pos = h.r_pos;
                size_t cnt = 0;
                if (down) {
                    for (long long j = 0; j < len; ++j) {  // resampling.rs:109-111
                        pos += out_rate;
                        if (pos >= in_rate) {
                            pos -= in_rate;
                            ++cnt;
                        }
                    }
                } else {
                    for (long long p = 0; p < len; ++p) {  // resampling.rs:247-266
                        while (pos < out_rate) {
                            ++cnt;
                            pos += in_rate;
                        }
                        pos -= out_rate;
                    }
                }
                h.r_pos = pos;
                a.n_new = cnt;
            } else {
                long long total_after;
                if (down) total_after = floordiv128(h.j0 + len, h.Q, h.P);  // outputs m with ceil(m*P/Q) <= J
                else total_after = ceildiv128(h.j0 + len, h.Q, h.P);        // q_p = ceil(p*Q/P), resampling.rs:249-266
                a.n_new = (size_t)(total_after - h.m0);
                const long long j1 = (h.j0 + len) % h.P;
                h.j0 = j1;
                h.m0 = down ? floordiv128(j1, h.Q, h.P) : ceildiv128(j1, h.Q, h.P);
            }
            a.pending_before = h.r_pending;
            const size_t ocl = d.output_chunk_len ? (size_t)d.output_chunk_len : 1;
            const size_t total = h.r_pending + a.n_new;
            a.out.chunk_len = ocl;
            a.out.n_chunks = total / ocl;
            a.out.rate = d.output_rate;
            h.r_pending = total - a.out.n_chunks * ocl;
            break;
        }
        default:
            return fail(RR_ERR_INVALID, "unknown stage kind");
    }
    *act = a;
    return RR_OK;
}

// An interrupt event reaches stage `h` (filters.rs:262-267, modulation.rs:133-138, chunks.rs:84-91,226-233).
// Returns the number of SamplesLost events the stage sends on top of it.
int stage_event(const rr_stage_desc& d, StageHost& h, bool* interrupt) {
    int lost = 0;
    switch (d.kind) {
        case RR_STAGE_RECHUNK:  // any event: the partial chunk is dropped and reported
            if (h.rc_pending > 0) {
                h.rc_pending = 0;
                lost = 1;
                *interrupt = true;
            }
            break;
        case RR_STAGE_OVERLAP:  // any event: history cleared, SamplesLost always sent
            h.ov_hist = 0;
            lost = 1;
            *interrupt = true;
            break;
        case RR_STAGE_FILTER:
            if (*interrupt) h.f_seg = 0;
            break;
        case RR_STAGE_FMDEMOD:
            if (*interrupt) h.fm_has_prev = false;
            break;
        default:
            break;
    }
    return lost;
}

// chunk lengths the device Filter takes
// the power-of-two chunk length the device kernels run a Filter of chunk length n with (n itself when it is one)
inline size_t filter_padded_len(size_t n) {
    size_t np = 32;
    while (np < n) np <<= 1;
    return np;
}
template <typename T> bool filter_len_supported(size_t n) {
    if (n < 1 || n > ((size_t)1 << 23)) return false;
    const size_t np = filter_padded_len(n);
    return rr::chain_os_supported<T>((int)np, 0, 0) || rr::big_os_supported<T>((int)np);
}
inline bool is_pow2(size_t n) { return n >= 2 && (n & (n - 1)) == 0; }

// what the device path cannot take is refused here, BEFORE a push changes any state (the dry run calls this)
int stage_supported(const rr_chain* c, const rr_stage_desc& d, const Shape& in) {
    if (in.n_chunks == 0 || in.chunk_len == 0) return RR_OK;
    const bool f32 = c->dtype == RR_C32;
    if (d.kind == RR_STAGE_FILTER) {
        const size_t n = in.chunk_len;
        if (!(f32 ? filter_len_supported<float>(n) : filter_len_supported<double>(n)))
            return fail(RR_ERR_UNSUPPORTED, "Filter: chunk length not supported by the device path");
    } else if (d.kind == RR_STAGE_FOURIER) {
        const int n = (int)std::min<size_t>(in.chunk_len, (size_t)1 << 30);
        const bool fft = f32 ? rr::fourier_fft_supported<float>(n) : rr::fourier_fft_supported<double>(n);
        if (!fft && in.chunk_len > (size_t)rr::kFourierDirectMax)
            return fail(RR_ERR_UNSUPPORTED, "Fourier: chunk lengths outside the FFT plans are limited to 4096 samples");
    }
    return RR_OK;
}

// output shape of a push without touching any state (capacity check, rr_chain_max_output); states (optional): every
// stage's host state as the push would leave it
int dry_shape(const rr_chain* c, const Shape& in, Shape* out, std::vector<StageHost>* states = nullptr) {
    std::vector<StageHost> hs;
    hs.reserve(c->st.size());
    for (const auto& s : c->st) hs.push_back(s.h);
    Shape sh = in;
    for (size_t i = 0; i < hs.size(); ++i) {
        StageAct a;
        RR_TRY(stage_supported(c, c->st[i].d, sh));
        RR_TRY(advance_stage(c->st[i].d, hs[i], sh, &a));
        if (a.lost) {
            bool intr = true;
            for (size_t j = i + 1; j < hs.size(); ++j) stage_event(c->st[j].d, hs[j], &intr);
        }
        sh = a.out;
    }
    *out = sh;
    if (states) *states = std::move(hs);
    return RR_OK;
}

template <typename T> struct TypeTag { using type = T; };
#define RR_DISPATCH(chain, T, ...)                     \
    do {                                               \
        if ((chain)->dtype == RR_C32) {                \
            using T = float;                           \
            __VA_ARGS__;                               \
        } else {                                       \
            using T = double;                          \
            __VA_ARGS__;                               \
        }                                              \
    } while (0)

rr::WindowFn make_window(int kind, double beta, rr_window_fn fn, void* user) {
    switch (kind) {
        case RR_WINDOW_RECTANGULAR:
            return [](double) { return 1.0; };
        case RR_WINDOW_CUSTOM:
            return [fn, user](double x) { return fn ? fn(user, x) : 1.0; };
        default:
            return [beta](double x) { return rr::kaiser_rel_with_beta(beta, x); };
    }
}

// upload a vector<complex<double>> as complex<T>
template <typename T> int upload_complex(DevBuf& buf, const std::vector<std::complex<double>>& v, cudaStream_t st) {
    RR_TRY(buf.ensure(v.size() * 2 * sizeof(T)));
    std::vector<T> tmp(v.size() * 2);
    for (size_t i = 0; i < v.size(); ++i) {
        tmp[2 * i] = (T)v[i].real();
        tmp[2 * i + 1] = (T)v[i].imag();
    }
    RR_CUDA(cudaMemcpyAsync(buf.p, tmp.data(), tmp.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    RR_CUDA(cudaStreamSynchronize(st));  // tmp is pageable and dies here
    return RR_OK;
}
template <typename T> int upload_real(DevBuf& buf, const std::vector<double>& v, cudaStream_t st) {
    RR_TRY(buf.ensure(v.size() * sizeof(T)));
    std::vector<T> tmp(v.size());
    for (size_t i = 0; i < v.size(); ++i) tmp[i] = (T)v[i];
    RR_CUDA(cudaMemcpyAsync(buf.p, tmp.data(), tmp.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    RR_CUDA(cudaStreamSynchronize(st));
    return RR_OK;
}

// ---- FreqShifter retune (transform.rs:318-340) ------------------------------
template <typename T> int nco_refresh(rr_chain* c, Stage& s, double sample_rate, bool rate_changed) {
    const int S = c->S;
    if (s.nco_h.empty()) s.nco_h.resize(S);
    s.nco_stage.resize(S);
    RR_TRY(s.nco_d.ensure(sizeof(rr::NcoStream) * (size_t)S));
    const bool all = rate_changed;
    if (!all && !s.any_shift_dirty) return RR_OK;
    const T tau = (T)6.283185307179586476925286766559;
    for (int i = 0; i < S; ++i) {
        NcoHost& h = s.nco_h[i];
        if (all || s.shift_dirty[i]) {
            // start_phase = arg(phase_vec[phase_idx]) in Flt, 0 when no table exists yet
            T start = (T)0;
            if (h.has_table) {
                const uint64_t prod = ((uint64_t)(h.numer < 0 ? -h.numer : h.numer) * (h.idx % (uint64_t)h.denom)) % (uint64_t)h.denom;
                const T iv = h.numer < 0 ? -(T)prod : (T)prod;
                const T ph = (T)h.start_phase + iv / (T)h.denom * tau;
                const T im = std::sin(ph), re = std::cos(ph);
                start = std::atan2(im, re);
            }
            int64_t numer = 0, denom = 1;
            if (!rr::freq_to_ratio(sample_rate, s.d.precision, s.shift[i], &numer, &denom))
                return fail(RR_ERR_INVALID, "FreqShifter: sample_rate / precision rounds to zero (Ratio::new panics)");
            if (denom <= 0 || denom >= (int64_t)1 << 31)
                return fail(RR_ERR_UNSUPPORTED, "FreqShifter: phase table length (sample_rate / precision) must be below 2^31");
            h.numer = numer;
            h.denom = denom;
            h.idx = 0;
            h.start_phase = (double)start;
            h.has_table = true;
            s.shift_dirty[i] = 0;
        }
        rr::NcoStream& d = s.nco_stage[i];
        const int64_t na = h.numer < 0 ? -h.numer : h.numer;
        d.numer_abs = (uint32_t)(na % h.denom);
        d.denom = (uint32_t)h.denom;
        d.idx = (uint32_t)(h.idx % (uint64_t)h.denom);
        d.sign = h.numer < 0 ? -1 : (h.numer > 0 ? 1 : 0);
        d.start_phase = h.start_phase;
    }
    s.any_shift_dirty = false;
    RR_CUDA(cudaMemcpyAsync(s.nco_d.p, s.nco_stage.data(), sizeof(rr::NcoStream) * (size_t)S, cudaMemcpyHostToDevice, c->stream));
    RR_CUDA(cudaStreamSynchronize(c->stream));
    return RR_OK;
}
void nco_host_advance(Stage& s, long long len) {
    for (auto& h : s.nco_h) h.idx = (h.idx + (uint64_t)len) % (uint64_t)h.denom;
}

// ---- Filter design + upload (filters.rs:184-238) ----------------------------
template <typename T> int filter_redesign(rr_chain* c, Stage& s, double sample_rate, size_t n) {
    s.taps_valid = false;  // until this design is complete, nothing may be built from the previous taps
    if (!filter_len_supported<T>(n)) return fail(RR_ERR_UNSUPPORTED, "Filter: chunk length not supported by the device path");
    const rr_stage_desc& d = s.d;
    if (!d.freq_resp) return fail(RR_ERR_INVALID, "Filter: freq_resp callback is null");
    rr_freq_resp_fn fn = d.freq_resp;
    void* user = d.freq_resp_user;
    rr::FreqResp f = [fn, user](int64_t bin, double freq) {
        double re = 0.0, im = 0.0;
        fn(user, bin, freq, &re, &im);
        return std::complex<double>(re, im);
    };
    rr::WindowFn w = make_window(d.window_kind, d.window_beta, d.window_fn, d.window_user);
    std::vector<std::complex<double>> H;
    if (!rr::design_filter_response(f, w, sample_rate, n, sizeof(T) == 4, &H, &s.taps))
        return fail(RR_ERR_UNSUPPORTED, "Filter: design failed");
    const size_t n_orig = n;
    s.f_np = filter_padded_len(n);
    if (s.f_np != n) {
        // z[k] = sum_{m<n} taps[m] x[k-m] on the kernels of chunk length f_np: the same taps, zero padded, in the second
        // half of a 2*f_np buffer (filters.rs:220-226 with n -> f_np)
        n = s.f_np;
        H.assign(2 * n, std::complex<double>(0.0, 0.0));
        for (size_t i = 0; i < n_orig; ++i) H[n + i] = s.taps[i];
        rr::fft_pow2(H, false);
        // ... and the reference's 1/(2 n^2) (filters.rs:186) goes with ITS inverse of 2n points; this one has 2*f_np
        const double fix = (double)n_orig / (double)n;
        for (auto& v : H) v *= fix;
        RR_TRY(s.zero_chunk.ensure(n * 2 * sizeof(T), true, c->stream));
    }
    const size_t N = 2 * n;
    if (rr::chain_os_supported<T>((int)n, 0, 0)) {
        std::vector<std::complex<double>> hp(N), tw;
        for (size_t k = 0; k < N; ++k) hp[(size_t)rr::chain_os_hperm_index<T>((int)n, (int)k)] = H[k];
        RR_TRY(upload_complex<T>(s.hperm, hp, c->stream));
        rr::make_twiddles(N, &tw);
        RR_TRY(upload_complex<T>(s.tw, tw, c->stream));
    } else if (rr::big_os_supported<T>((int)n)) {
        int Na = 0, Nb = 0;
        rr::big_os_shape<T>((int)n, &Na, &Nb);
        std::vector<std::complex<double>> hp(N), tw;
        for (size_t k = 0; k < N; ++k) hp[(size_t)rr::big_os_hperm_index<T>((int)n, (long long)k)] = H[k];
        RR_TRY(upload_complex<T>(s.big_h, hp, c->stream));
        rr::make_twiddles(N, &tw);
        RR_TRY(upload_complex<T>(s.tw, tw, c->stream));
        rr::make_twiddles((size_t)Na, &tw);
        RR_TRY(upload_complex<T>(s.big_twA, tw, c->stream));
        rr::make_twiddles((size_t)Nb, &tw);
        RR_TRY(upload_complex<T>(s.big_twB, tw, c->stream));
        if (rr::long_os_supported((int)n)) {
            std::vector<std::complex<double>> full, small((size_t)rr::long_os_twc_size<T>((int)n));
            rr::make_twiddles(N, &full);
            for (size_t i = 0; i < small.size(); ++i) small[i] = full[(size_t)rr::long_os_twc_exponent<T>((int)n, (int)i)];
            RR_TRY(upload_complex<T>(s.big_twC, small, c->stream));
        }
    } else {
        return fail(RR_ERR_UNSUPPORTED, "Filter: chunk length not supported by the device path");
    }
    const size_t hb = (size_t)c->S * 2 * n_orig * 2 * sizeof(T);
    RR_TRY(s.hist2[0].ensure(hb));
    RR_TRY(s.hist2[1].ensure(hb));
    s.taps_valid = true;
    return RR_OK;
}

// ---- resampler taps (resampling.rs:82-101, :216-236) -------------------------
template <typename T> int resampler_redesign(rr_chain* c, Stage& s, double in_rate) {
    const rr_stage_desc& d = s.d;
    const bool down = d.kind == RR_STAGE_DOWNSAMPLE;
    const int L = s.h.r_L;
    const double margin = down ? (d.output_rate - d.bandwidth) / 2.0 : (in_rate - d.bandwidth) / 2.0;
    const double ratio = down ? d.output_rate / in_rate : in_rate / d.output_rate;
    const double null_bin = (double)L * margin / (down ? in_rate : d.output_rate);
    rr::design_resampler_taps((size_t)L, ratio, null_bin, &s.ir_host);
    RR_TRY(upload_real<T>(s.ir, s.ir_host, c->stream));
    s.ir_host_flt.resize(s.ir_host.size());
    for (size_t i = 0; i < s.ir_host.size(); ++i) s.ir_host_flt[i] = (double)(T)s.ir_host[i];
    // ring buffer / accumulators restart at zero (resampling.rs:99-101, :234-236)
    const size_t state_len = down ? (size_t)(L > 1 ? L - 1 : 1) : (size_t)L;
    const size_t tb = (size_t)c->S * state_len * 2 * sizeof(T);
    for (int k = 0; k < 2; ++k) {
        RR_TRY(s.tail[k].ensure(tb));
        RR_CUDA(cudaMemsetAsync(s.tail[k].p, 0, tb, c->stream));
    }
    s.tail_cur = 0;
    s.ztail_stale = false;
    s.poly_valid = false;
    s.poly_tried = false;
    return RR_OK;
}

// make room for `need` samples per stream in both output staging buffers of a
// resampler, preserving the `keep` pending samples of the current one
template <typename T> int obuf_reserve(rr_chain* c, Stage& s, size_t need, size_t keep) {
    if (need <= s.obuf_cap && s.obuf[0].p && s.obuf[1].p) return RR_OK;
    size_t cap = need + need / 2 + 16;
    const size_t bytes = (size_t)c->S * cap * 2 * sizeof(T);
    DevBuf nb0, nb1;
    RR_TRY(nb0.ensure(bytes));
    RR_TRY(nb1.ensure(bytes));
    if (keep && s.obuf[s.obuf_cur].p) {
        RR_LAUNCH(1, rr::launch_copy2d<T>(s.obuf[s.obuf_cur].p, (long long)s.obuf_cap, nb0.p, (long long)cap, (long long)keep, c->S,
                                          c->stream));
        RR_CUDA(cudaStreamSynchronize(c->stream));
    }
    s.obuf[0].release();
    s.obuf[1].release();
    s.obuf[0] = nb0;
    s.obuf[1] = nb1;
    s.obuf_cur = 0;
    s.obuf_cap = cap;
    return RR_OK;
}

template <typename T> int out_reserve(rr_chain* c, Stage& s, size_t need) {
    if (need <= s.out_cap && s.out.p) return RR_OK;
    RR_TRY(s.out.ensure((size_t)c->S * need * 2 * sizeof(T)));
    s.out_cap = need;
    return RR_OK;
}

struct Dest {
    void* p = nullptr;
    long long stride = 0;
};

// chooses where a stage writes: the caller's buffer when it is the last stage
template <typename T> int pick_dest(rr_chain* c, Stage& s, bool last, void* user_out, long long user_stride, size_t len, Dest* d) {
    if (last) {
        d->p = user_out;
        d->stride = user_stride;
        return RR_OK;
    }
    RR_TRY(out_reserve<T>(c, s, len));
    d->p = s.out.p;
    d->stride = (long long)s.out_cap;
    return RR_OK;
}

// after a resampler wrote n_new samples behind `pending_before` ones in its
// staging buffer: hand whole chunks downstream, keep the remainder
template <typename T>
int resampler_emit(rr_chain* c, Stage& s, const StageAct& a, bool last, void* user_out, long long user_stride, View* next,
                   bool direct_done = false) {
    const size_t emit = a.out.len();
    const size_t total = a.pending_before + a.n_new;
    DevBuf& cur = s.obuf[s.obuf_cur];
    DevBuf& other = s.obuf[s.obuf_cur ^ 1];
    const size_t rem = total - emit;
    if (direct_done) {
        // the kernel wrote the new samples to user_out / `other` itself: only the samples that were pending
        // before this push are still in `cur`
        if (a.pending_before > 0)
            RR_LAUNCH(1, rr::launch_copy2d<T>(cur.p, (long long)s.obuf_cap, user_out, user_stride, (long long)a.pending_before, c->S, c->stream));
        next->sh = a.out;
        next->p = user_out;
        next->stride = user_stride;
        s.obuf_cur ^= 1;
        return RR_OK;
    }
    if (rem > 0 && emit > 0) {
        const char* src = (const char*)cur.p + emit * 2 * sizeof(T);
        RR_LAUNCH(1, rr::launch_copy2d<T>(src, (long long)s.obuf_cap, other.p, (long long)s.obuf_cap, (long long)rem, c->S, c->stream));
    }
    next->sh = a.out;
    if (last) {
        if (emit > 0)
            RR_LAUNCH(1, rr::launch_copy2d<T>(cur.p, (long long)s.obuf_cap, user_out, user_stride, (long long)emit, c->S, c->stream));
        next->p = user_out;
        next->stride = user_stride;
    } else {
        next->p = cur.p;
        next->stride = (long long)s.obuf_cap;
    }
    if (emit > 0) s.obuf_cur ^= 1;  // the remainder (possibly empty) now lives in `other`
    return RR_OK;
}

// ---------------------------------------------------------------------------
// Filter (+ Downsampler) execution.  Three device paths:
//   poly      NCO -> Filter -> Downsampler fused, polyphase (rr_poly.cuh): the
//             throughput path; needs two chunks of in-segment history
//   fused_os  NCO -> overlap-save (-> FIR decimator) per stream in one CTA
//             (rr_chain_os.cuh): the stateful path, any segment position
//   big_os    four-step FFT overlap-save for long chunks (rr_big_os.cu)
// State shared by all of them: hist2 (two post-NCO chunks) on the filter stage
// and tail (the last L-1 filter outputs) on the downsampler stage.
// ---------------------------------------------------------------------------
struct FilterIo {
    const void* in = nullptr;  // pushed samples (pre-NCO when nco != nullptr)
    long long in_stride = 0;
    size_t n = 0, n_chunks = 0;
    Stage* nco = nullptr;
    bool shared = false;  // `in` is the row of a shared push that every stream reads (in_stride 0, S > 1)
};

// run the stand-alone NCO kernel over chunks [c0, c0+k) into the NCO stage's buffer
template <typename T> int materialize_nco(rr_chain* c, Stage& nco, const FilterIo& io, size_t c0, size_t k, const void** out, long long* stride) {
    const size_t len = k * io.n;
    RR_TRY(out_reserve<T>(c, nco, len));
    const char* src = (const char*)io.in + c0 * io.n * 2 * sizeof(T);
    RR_LAUNCH(1, rr::launch_freqshift<T>(src, io.in_stride, nco.out.p, (long long)nco.out_cap, (long long)len, c->S,
                                         (const rr::NcoStream*)nco.nco_d.p, (long long)(c0 * io.n), c->stream));
    *out = nco.out.p;
    *stride = (long long)nco.out_cap;
    return RR_OK;
}

// Overlap-save over the first k chunks of the push; history for chunk 0 is
// hist2's newer half; `fih`: chunk 0 only primes the filter (filters.rs:240,260).
// Writes (k - fih) * n filter outputs to dst.
template <typename T>
int run_os(rr_chain* c, Stage& s, const FilterIo& io, size_t k, bool fih, void* dst, long long dst_stride, const void* hist_override = nullptr,
           long long hist_stride_override = 0);

// Chunk lengths that are not a power of two (filters.rs:227-228 plans any length): the filter is
// z[t] = sum_{m<n} taps[m] x[t-m], so it can run on the kernels of the next power of two f_np with the taps zero
// padded.  [history chunk | pushed chunks] is staged contiguously (mixed, when an NCO is folded in), cut into chunks of
// f_np behind a zero chunk, transformed, and the outputs of the pushed samples are copied out.
template <typename T>
int run_os_padded(rr_chain* c, Stage& s, const FilterIo& io, size_t k, bool fih, void* dst, long long dst_stride) {
    const size_t n = io.n, np = s.f_np, esz = 2 * sizeof(T);
    const int S = c->S;
    const size_t n_hist = fih ? 0 : n;
    const size_t Ls = n_hist + k * n;            // staged samples per stream
    if (Ls <= n) return RR_OK;                    // nothing to emit
    const size_t nch = (Ls + np - 1) / np;        // chunks of f_np
    const size_t stride = nch * np;
    RR_TRY(s.stg_in.ensure((size_t)S * stride * esz));
    RR_TRY(s.stg_out.ensure((size_t)S * stride * esz));
    char* stg = (char*)s.stg_in.p;
    if (n_hist) {
        const char* hist_newer = (const char*)s.hist2[s.hist_cur].p + n * esz;
        RR_LAUNCH(1, rr::launch_copy2d<T>(hist_newer, (long long)(2 * n), stg, (long long)stride, (long long)n, S, c->stream));
    }
    if (io.nco) {
        RR_LAUNCH(1, rr::launch_freqshift<T>(io.in, io.in_stride, stg + n_hist * esz, (long long)stride, (long long)(k * n), S,
                                             (const rr::NcoStream*)io.nco->nco_d.p, 0, c->stream));
    } else {
        RR_LAUNCH(1, rr::launch_copy2d<T>(io.in, io.in_stride, stg + n_hist * esz, (long long)stride, (long long)(k * n), S, c->stream));
    }
    if (stride > Ls)
        RR_CUDA(cudaMemset2DAsync(stg + Ls * esz, stride * esz, 0, (stride - Ls) * esz, (size_t)S, c->stream));
    FilterIo pio;
    pio.in = stg;
    pio.in_stride = (long long)stride;
    pio.n = np;
    pio.n_chunks = nch;
    pio.nco = nullptr;
    RR_TRY(run_os<T>(c, s, pio, nch, false, s.stg_out.p, (long long)stride, s.zero_chunk.p, 0));
    // staged index t holds the filter output of staged sample t: the pushed samples' outputs start at index n
    RR_LAUNCH(1, rr::launch_copy2d<T>((const char*)s.stg_out.p + n * esz, (long long)stride, dst, dst_stride, (long long)(Ls - n), S, c->stream));
    return RR_OK;
}

template <typename T>
int run_os(rr_chain* c, Stage& s, const FilterIo& io, size_t k, bool fih, void* dst, long long dst_stride, const void* hist_override,
           long long hist_stride_override) {
    const size_t n = io.n;
    const int S = c->S;
    if (k == 0) return RR_OK;
    if (!hist_override && s.f_np != 0 && s.f_np != n) return run_os_padded<T>(c, s, io, k, fih, dst, dst_stride);
    const char* hist_newer = hist_override ? (const char*)hist_override : (const char*)s.hist2[s.hist_cur].p + n * 2 * sizeof(T);
    const long long hist_stride = hist_override ? hist_stride_override : (long long)(2 * n);
    if (rr::chain_os_supported<T>((int)n, 0, 0)) {
        rr::ChainOsArgs<T> a{};
        a.in = io.in;
        a.in_stride = io.in_stride;
        a.n_chunks = (int)k;
        a.first_is_history = fih ? 1 : 0;
        a.emit = 1;
        a.hist_in = hist_newer;
        a.hist_stride = hist_stride;
        a.hist_out = nullptr;
        a.hperm = s.hperm.p;
        a.twN = s.tw.p;
        a.nco = io.nco ? (const rr::NcoStream*)io.nco->nco_d.p : nullptr;
        a.nco_offset = 0;
        a.out = dst;
        a.out_stride = dst_stride;
        int parts = 1;
        const int total = a.n_chunks - a.first_is_history;
        if (total > 1) {
            const int want = (2 * c->ctx->sm_count + S - 1) / S;
            parts = want < total ? want : total;
            if (parts < 1) parts = 1;
        }
        RR_TIMED_LAUNCH(c, "k_chain_os<epi=none>", 1, rr::launch_chain_os<T>((int)n, 0, S, parts, a, c->stream));
        return RR_OK;
    }
    if (!rr::big_os_supported<T>((int)n)) return fail(RR_ERR_UNSUPPORTED, "Filter: chunk length not supported by the device path");
    const void* src = io.in;
    long long src_stride = io.in_stride;
    if (io.nco) RR_TRY(materialize_nco<T>(c, *io.nco, io, 0, k, &src, &src_stride));  // the four-step kernels take mixed samples
    const size_t N = 2 * n;
    const size_t first = fih ? 1 : 0;  // first chunk that produces output
    const size_t n_blocks = k - first;
    if (n_blocks == 0) return RR_OK;
    const size_t esz = 2 * sizeof(T);
    // the three kernels of a launch group exchange their blocks through `scratch`.  Measured (256 x 8 blocks of 2^17
    // points f32, 16 x 4 blocks of 2^20 points f64): groups small enough to keep the scratch in L2 (24-96 MiB) are
    // 15-30 % SLOWER than one large launch on one stream -- small launches, and their tails, cost more than the L2 hits
    // save -- and level with it when the groups go round 2-6 side streams (commit 2f092e5 has that form); the kernels sit
    // on the fp32 / fp64 pipe right behind the HBM bound (DESIGN 4.3).  So the bound only limits the memory taken (2 GiB)
    size_t max_blocks = c->big_os_scratch_bytes / (N * 2 * sizeof(T));
    if (max_blocks < 1) max_blocks = 1;
    const size_t sg = std::min<size_t>((size_t)S, max_blocks);  // streams per launch group
    size_t per_launch = max_blocks / sg;
    if (per_launch < 1) per_launch = 1;
    if (per_launch > n_blocks) per_launch = n_blocks;
    RR_TRY(s.big_scratch.ensure(sg * per_launch * N * 2 * sizeof(T)));
    for (size_t s0 = 0; s0 < (size_t)S; s0 += sg) {
        const int sn = (int)std::min(sg, (size_t)S - s0);
        for (size_t b0 = 0; b0 < n_blocks; b0 += per_launch) {
            const size_t nb = std::min(per_launch, n_blocks - b0);
            rr::BigOsArgs<T> a{};
            a.in = (const char*)src + s0 * (size_t)src_stride * esz;
            a.in_stride = src_stride;
            a.hist = hist_newer + s0 * (size_t)hist_stride * esz;
            a.hist_stride = hist_stride;
            a.first_chunk = (int)(first + b0);
            a.n_blocks = (int)nb;
            a.scratch = s.big_scratch.p;
            a.hbig = s.big_h.p;
            a.twN = s.tw.p;
            a.twA = s.big_twA.p;
            a.twB = s.big_twB.p;
            a.twC = s.big_twC.p;
            a.out = (char*)dst + (s0 * (size_t)dst_stride + b0 * n) * esz;
            a.out_stride = dst_stride;
            RR_TIMED_LAUNCH(c, "k_big_os(3 kernels)", 3, rr::launch_big_os<T>((int)n, sn, a, c->stream));
        }
    }
    return RR_OK;
}

// rebuild the downsampler's tail (last L-1 filter outputs) from the filter's hist2
template <typename T> int regen_ztail(rr_chain* c, Stage& f, Stage& ds) {
    if (!ds.ztail_stale) return RR_OK;
    const size_t n = f.h.f_n;
    const int L = ds.h.r_L;
    if (L > 1) {
        DevBuf& tmp = f.ztmp;
        RR_TRY(tmp.ensure((size_t)c->S * n * 2 * sizeof(T)));
        FilterIo io;
        io.in = f.hist2[f.hist_cur].p;
        io.in_stride = (long long)(2 * n);
        io.n = n;
        io.n_chunks = 2;
        io.nco = nullptr;
        RR_TRY(run_os<T>(c, f, io, 2, true, tmp.p, (long long)n));
        const char* src = (const char*)tmp.p + (n - (size_t)(L - 1)) * 2 * sizeof(T);
        RR_LAUNCH(1, rr::launch_copy2d<T>(src, (long long)n, ds.tail[ds.tail_cur].p, (long long)(L - 1), (long long)(L - 1), c->S, c->stream));
    }
    ds.ztail_stale = false;
    return RR_OK;
}

// k_fused reads its coefficient table from constant memory: a few slots per device, owned by Downsampler stages
std::mutex g_slot_mu;
const void* g_slot_owner[16][8] = {};
int fused_slot_acquire(int device, const void* owner) {
    if (device < 0 || device >= 16) return -1;
    std::lock_guard<std::mutex> lk(g_slot_mu);
    const int n = std::min(8, rr::fused_coef_slots());
    for (int i = 0; i < n; ++i)
        if (g_slot_owner[device][i] == owner) return i;
    for (int i = 0; i < n; ++i)
        if (!g_slot_owner[device][i]) {
            g_slot_owner[device][i] = owner;
            return i;
        }
    return -1;
}
void fused_slot_release(int device, const void* owner) {
    if (device < 0 || device >= 16) return;
    std::lock_guard<std::mutex> lk(g_slot_mu);
    for (int i = 0; i < 8; ++i)
        if (g_slot_owner[device][i] == owner) g_slot_owner[device][i] = nullptr;
}

constexpr int kFrontQRank = 16;  // columns of the Q > 1 front end (two rounds of k_poly's G = 8)

// (re)build the polyphase tables for the pair (filter f, downsampler ds)
template <typename T> int poly_prepare(rr_chain* c, Stage& f, Stage& ds) {
    if (ds.poly_tried) return RR_OK;
    ds.poly_tried = true;
    ds.poly_valid = false;
    ds.poly2_valid = false;
    ds.front_valid = false;
    ds.frontq_valid = false;
    ds.fused_valid = false;
    if (!f.taps_valid) return RR_OK;
    const long long P = ds.h.P, Q = ds.h.Q;
    const long long n = (long long)f.h.f_n, L = ds.h.r_L;
    if (Q > 4 || P < 2 || L - 1 > n || L < 2) return RR_OK;
    const long long Lmax = (n + L - 2) / P;
    int bestK = 0;
    double best = 0.0;
    for (int K : {256, 512, 1024}) {
        const long long V = K - 1 - Lmax;
        if (V < K / 4) continue;
        double cost = (5.0 * std::log2((double)K) + 8.0 * (double)Q + 8.0) * (double)K / (double)V;
        if (K == 1024) cost *= 1.1;  // larger working set: only when clearly better
        if (bestK == 0 || cost < best) {
            bestK = K;
            best = cost;
        }
    }
    if (bestK == 0) return RR_OK;
    const size_t tab_bytes = (size_t)(Q * P) * (size_t)bestK * 2 * sizeof(T);
    if (tab_bytes > ((size_t)512 << 20)) return RR_OK;
    const double e8 = (double)P / (8.0 * (double)((P + 7) / 8)), e10 = (double)P / (10.0 * (double)((P + 9) / 10));
    const int G = e10 > e8 + 1e-9 ? 10 : 8;
    if (!rr::poly_supported<T>(bestK, (int)Q, G)) return RR_OK;
    if (rr::poly_smem_bytes<T>(bestK, (int)Q, G, 1) > (size_t)220 * 1024) return RR_OK;
    std::vector<std::complex<double>> tab, perm;
    const int lm = rr::design_poly_tables(f.taps, ds.ir_host_flt, P, Q, bestK, &tab);
    if (lm != (int)Lmax) return fail(RR_ERR_INVALID, "internal: polyphase reach mismatch");
    // f.taps carry the 1/(2n) of the reference's unnormalised 2n-point inverse (filters.rs:186); the
    // kernel's K-point forward/inverse pair is unnormalised too: rescale by 2n / K
    const double scale = 2.0 * (double)n / (double)bestK;
    // device layout [q][round][bin position][g]: the G branches of a round sit side by side (one
    // coalesced read per bin), branches past P are zero
    const long long NR = (P + G - 1) / G;
    perm.assign((size_t)(Q * NR) * (size_t)bestK * (size_t)G, std::complex<double>(0.0, 0.0));
    for (long long q = 0; q < Q; ++q)
        for (long long p = 0; p < P; ++p) {
            const long long r = p / G, gg = p % G;
            for (int k = 0; k < bestK; ++k) {
                const size_t pos = (size_t)rr::poly_hperm_index<T>(bestK, k);
                perm[(((size_t)(q * NR + r)) * bestK + pos) * G + gg] = tab[(size_t)(q * P + p) * bestK + k] * scale;
            }
        }
    RR_TRY(upload_complex<T>(ds.gtab, perm, c->stream));
    std::vector<std::complex<double>> tw;
    rr::make_twiddles((size_t)bestK, &tw);
    RR_TRY(upload_complex<T>(ds.twK, tw, c->stream));
    ds.poly_K = bestK;
    ds.poly_G = G;
    ds.poly_Lmax = (int)Lmax;
    ds.poly_V = (int)(bestK - 1 - Lmax);
    ds.poly_valid = true;

    // Q > 1, complex f32: the Q phase matrices factored together (rr_design.h: design_rank_tables_q).  The front end
    // (16 or 32 columns: k_front for even P <= 254, k_front_wide for any P) is shared by the phases; the low-rate part is
    // k_poly on u as a stream of that many branches with one table per phase -- 16 / 32 instead of P forward transforms
    // per block
    if (std::is_same<T, float>::value && Q > 1 && c->allow_front && P > 2 * kFrontQRank && rr::poly_supported<T>(bestK, (int)Q, 8) &&
        Lmax + 2 <= bestK) {
        constexpr int RMAX = 2 * kFrontQRank;
        std::vector<double> acf;
        std::vector<std::complex<double>> bq;
        int rank = 0;
        double disc = 0.0;
        const int lmq = rr::design_rank_tables_q(f.taps, ds.ir_host_flt, P, Q, bestK, 2.0e-8, RMAX, &rank, &acf, &bq, &disc);
        const int cols = rank <= kFrontQRank ? kFrontQRank : RMAX;
        const bool narrow = cols == kFrontQRank && rr::front_supported(kFrontQRank, P);
        if (rank > 0 && lmq == (int)Lmax && (narrow || rr::front_wide_supported(cols, P))) {
            std::vector<double> ac((size_t)P * cols);
            for (long long p = 0; p < P; ++p)
                for (int cc = 0; cc < cols; ++cc) ac[(size_t)p * cols + cc] = acf[(size_t)p * RMAX + cc];
            RR_TRY(upload_real<float>(ds.acoef_q, ac, c->stream));
            constexpr int GQ = 8;
            const long long NRq = cols / GQ;
            perm.assign((size_t)(Q * NRq) * (size_t)bestK * (size_t)GQ, std::complex<double>(0.0, 0.0));
            for (long long q = 0; q < Q; ++q)
                for (int cc = 0; cc < cols; ++cc) {
                    const long long r = cc / GQ, gg = cc % GQ;
                    for (int k = 0; k < bestK; ++k) {
                        const size_t pos = (size_t)rr::poly_hperm_index<T>(bestK, k);
                        perm[(((size_t)(q * NRq + r)) * bestK + pos) * GQ + gg] = bq[((size_t)q * RMAX + cc) * bestK + k] * scale;
                    }
                }
            RR_TRY(upload_complex<T>(ds.gtab_q, perm, c->stream));
            ds.frontq_rank = rank;
            ds.frontq_cols = cols;
            ds.frontq_wide = !narrow;
            ds.frontq_discarded = disc;
            ds.frontq_valid = true;
        }
    }

    // the packed-fp32 / TMA kernel: complex f32, integer decimation, K = 512
    if (std::is_same<T, float>::value && c->allow_poly2 && rr::poly2_supported(512, P, Q) && 511 - Lmax >= 128) {
        const int K2 = 512, G2 = rr::poly2_pick_G(P);
        if (bestK != K2) rr::design_poly_tables(f.taps, ds.ir_host_flt, P, Q, K2, &tab);
        const double scale2 = 2.0 * (double)n / (double)K2;
        const long long NR2 = (P + G2 - 1) / G2;
        perm.assign((size_t)NR2 * (size_t)K2 * (size_t)G2, std::complex<double>(0.0, 0.0));
        for (long long p = 0; p < P; ++p)
            for (int k = 0; k < K2; ++k)
                perm[(size_t)rr::poly2_table_index(G2, (int)(p / G2), (int)(p % G2), k)] = tab[(size_t)p * K2 + k] * scale2;
        RR_TRY(upload_complex<T>(ds.gtab2, perm, c->stream));
        if (bestK != K2) {
            rr::make_twiddles((size_t)K2, &tw);
            RR_TRY(upload_complex<T>(ds.twK2, tw, c->stream));
        }
        ds.poly2_tw_own = bestK != K2;
        ds.poly2_G = G2;
        ds.poly2_V = (int)(K2 - 1 - Lmax);
        ds.poly2_valid = true;

        // rank-reduced form: the P x (Lmax+1) matrix of the fused filter to below f32 rounding
        constexpr int RK = 10;
        if (c->allow_front && rr::front_supported(RK, P) && rr::poly2_supported(K2, RK, 1)) {
            std::vector<double> acf;
            std::vector<std::complex<double>> bfft;
            int rank = 0;
            double disc = 0.0;
            const int lm2 = rr::design_rank_tables(f.taps, ds.ir_host_flt, P, K2, 2.0e-8, RK, &rank, &acf, &bfft, &disc);
            if (rank > 0 && lm2 == (int)Lmax) {
                std::vector<double> ac((size_t)P * RK);
                for (long long p = 0; p < P; ++p)
                    for (int cc = 0; cc < RK; ++cc) ac[(size_t)(((p / 2) * 2 + (p & 1)) * RK + cc)] = acf[(size_t)p * RK + cc];
                RR_TRY(upload_real<float>(ds.acoef, ac, c->stream));
                perm.assign((size_t)K2 * (size_t)RK, std::complex<double>(0.0, 0.0));
                for (int cc = 0; cc < RK; ++cc)
                    for (int k = 0; k < K2; ++k) perm[(size_t)rr::poly2_table_index(RK, 0, cc, k)] = bfft[(size_t)cc * K2 + k] * scale2;
                RR_TRY(upload_complex<T>(ds.gtab3, perm, c->stream));
                ds.front_rank = rank;
                ds.front_discarded = disc;
                ds.front_valid = true;
                // the fused kernel takes the same coefficients through constant memory
                if (c->allow_fused && rr::fused_supported(RK, P, (int)Lmax)) {
                    const int slot = fused_slot_acquire(c->ctx->device, &ds);
                    if (slot >= 0) {
                        RR_CUDA(rr::fused_upload_coef(slot, (const float*)ds.acoef.p, (int)P, c->stream));
                        ds.fused_slot = slot;
                        ds.fused_valid = true;
                    }
                }
            }
        }
    }
    return RR_OK;
}

// ---- resamplers at rates that are not integer valued ---------------------------------------------------------
// The firing instants come from the reference's own f64 `pos` recurrence, replayed on the host for this push
// (StageAct::pos0 = pos before the push), and are uploaded as index tables.
template <typename T>
int downsample_indexed(rr_chain* c, Stage& ds, const StageAct& a, const void* in, long long in_stride, long long len, void* out,
                       long long out_stride) {
    const double in_rate = ds.h.r_in_rate, out_rate = ds.d.output_rate;
    std::vector<int> fire;
    fire.reserve(a.n_new);
    double pos = a.pos0;
    for (long long j = 0; j < len; ++j) {  // resampling.rs:109-111
        pos += out_rate;
        if (pos >= in_rate) {
            pos -= in_rate;
            fire.push_back((int)j);
        }
    }
    if (fire.size() != a.n_new) return fail(RR_ERR_INVALID, "internal: indexed downsampler count mismatch");
    RR_TRY(ds.idx_a.ensure(std::max<size_t>(fire.size(), 1) * sizeof(int)));
    if (!fire.empty()) RR_CUDA(cudaMemcpyAsync(ds.idx_a.p, fire.data(), fire.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    RR_CUDA(cudaStreamSynchronize(c->stream));  // `fire` is pageable and dies here
    RR_LAUNCH(2, rr::launch_downsample_indexed<T>(in, in_stride, len, ds.tail[ds.tail_cur].p, ds.tail[ds.tail_cur ^ 1].p, (const T*)ds.ir.p,
                                                  ds.h.r_L, (const int*)ds.idx_a.p, (long long)fire.size(), out, out_stride, c->S, c->stream));
    ds.tail_cur ^= 1;
    return RR_OK;
}
template <typename T>
int upsample_indexed(rr_chain* c, Stage& us, const StageAct& a, const void* in, long long in_stride, long long len, void* out,
                     long long out_stride) {
    const double in_rate = us.h.r_in_rate, out_rate = us.d.output_rate;
    const int L = us.h.r_L;
    std::vector<int> qpos((size_t)len);
    double pos = a.pos0;
    long long q = 0;
    for (long long p = 0; p < len; ++p) {  // resampling.rs:239-266: input p lands at the next cell to be emitted
        qpos[(size_t)p] = (int)q;
        while (pos < out_rate) {
            ++q;
            pos += in_rate;
        }
        pos -= out_rate;
    }
    if ((size_t)q != a.n_new) return fail(RR_ERR_INVALID, "internal: indexed upsampler count mismatch");
    // cnt[i] = number of inputs with qpos <= i, i < n_new + L
    std::vector<int> cnt((size_t)q + (size_t)L);
    {
        size_t p = 0;
        for (size_t i = 0; i < cnt.size(); ++i) {
            while (p < qpos.size() && (size_t)qpos[p] <= i) ++p;
            cnt[i] = (int)p;
        }
    }
    RR_TRY(us.idx_a.ensure(std::max<size_t>(qpos.size(), 1) * sizeof(int)));
    RR_TRY(us.idx_b.ensure(std::max<size_t>(cnt.size(), 1) * sizeof(int)));
    if (!qpos.empty()) RR_CUDA(cudaMemcpyAsync(us.idx_a.p, qpos.data(), qpos.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    if (!cnt.empty()) RR_CUDA(cudaMemcpyAsync(us.idx_b.p, cnt.data(), cnt.size() * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    RR_CUDA(cudaStreamSynchronize(c->stream));
    RR_LAUNCH(1, rr::launch_upsample_indexed<T>(in, in_stride, len, us.tail[us.tail_cur].p, us.tail[us.tail_cur ^ 1].p, (const T*)us.ir.p, L,
                                                (const int*)us.idx_a.p, (const int*)us.idx_b.p, q, out, out_stride, c->S, c->stream));
    us.tail_cur ^= 1;
    return RR_OK;
}

// Filter stage `f` (with optional folded NCO) followed by Downsampler `ds`:
// consumes the whole push, leaves new outputs behind ds's pending samples.
// `direct` (optional): the Downsampler is the chain's last stage -- when the whole push goes through k_poly2, its
// outputs are written straight to the caller's buffer (whole output chunks) and to the other obuf (the part
// behind them), and *direct->done tells resampler_emit that only the old pending samples are left to copy.
struct DirectOut {
    void* user_out = nullptr;
    long long user_stride = 0;
    bool done = false;
};

// ---- the polyphase part of run_filter_down ----------------------------------------------------------------------
// What its routes share: the chunks [ca, n_chunks) of the push, whose filter outputs fire the Downsampler's outputs
// m_lo..m_hi (1-based, counted with the reduced counters).  Filter output k aligns with push sample k; the kernels
// read the (mixed on the fly) push chunks before the part, or hist2 below offset 0.
struct PolyPart {
    rr_chain* c;
    Stage& f;
    Stage& ds;
    const FilterIo& io;
    const StageAct& da;
    DirectOut* direct;
    long long P, Q;       // in/out = P/Q reduced
    long long J0, m0;     // decimator counters referred to push sample 0 (J0 may be negative)
    long long m_lo, m_hi;
    long long I_lo, I_hi;  // low-rate indices of outputs m_lo and m_hi
    long long len, n;     // pushed samples per stream, Filter chunk length
    const rr::NcoStream* nco;
    void* obase;          // output m goes to obase[m - m0 - 1] (rows ostride apart)
    long long ostride;
    bool tma_ok;          // (complex f32) the pushed samples can be read by TMA: rr::tma_input_ok
    bool whole;           // the whole push is polyphase (no stateful chunks in front)
    bool kept;            // whole, and the u rows the previous push kept are usable
};

// The Filter's next history is the last 2n mixed samples of the push, from push offset len - 2n.  A front end whose
// rows cover push offsets [cover_lo, cover_hi) writes it, from max(len - 2n, 0) up to its last row, when those rows
// reach back to that start; k_hist2_update copies the rest (Stage::hist_fused_*).  (A push shorter than 2n keeps the
// end of the old history in front: those entries, [0, 2n - len), are always k_hist2_update's.)
template <typename A> bool next_history(const PolyPart& p, long long cover_lo, long long cover_hi, A* a) {
    Stage& f = p.f;
    f.hist_fused_jlo = -1;
    f.hist_fused_jfirst = 0;
    const long long hfrom = p.len - 2 * p.n, hstart = std::max<long long>(hfrom, 0);
    if (cover_lo > hstart || cover_hi <= hstart) return false;
    a->hist_out = f.hist2[f.hist_cur ^ 1].p;
    a->hist_from = hfrom;
    a->hist_stride = 2 * p.n;
    f.hist_fused_jlo = cover_hi - hfrom;
    f.hist_fused_jfirst = hstart - hfrom;
    return true;
}

// Direct output (complex f32): new output o lands at emitted position pending_before + o, so the outputs that complete
// the caller's chunks go to the caller's buffer and the ones behind them (from out_split) to the other obuf
template <typename A> void direct_split(const PolyPart& p, A* a) {
    const long long emit = (long long)p.da.out.len();
    if (!p.direct || !p.direct->user_out || emit < (long long)p.da.pending_before || emit <= 0) return;
    a->out = (char*)p.direct->user_out + p.da.pending_before * 2 * sizeof(float);
    a->out_stride = p.direct->user_stride;
    a->out2 = p.ds.obuf[p.ds.obuf_cur ^ 1].p;
    a->out2_stride = p.ostride;
    a->out_split = emit - (long long)p.da.pending_before;
    p.direct->done = true;
}

// k_poly2 blocks per group (one round of inverse transforms; bounded by shared memory) and groups per CTA half: as many
// as keep the grid at two CTAs per SM or more, balanced
void poly2_grid(rr::PolyArgs<float>* a, int G, int S, int sm_count) {
    int nbpc = std::min(G, a->n_blocks);
    while (nbpc > 1 && rr::poly2_smem_bytes(G, nbpc) > (size_t)226 * 1024) --nbpc;
    const long long ctas_y = (S + 1) / 2;
    while (nbpc > 1 && ctas_y * ((a->n_blocks + nbpc - 1) / nbpc) < 2LL * sm_count) --nbpc;
    const int ngroups = (a->n_blocks + nbpc - 1) / nbpc;
    a->nbpc = (a->n_blocks + ngroups - 1) / ngroups;
    int ngrp = ngroups;
    while (ngrp > 1 && ctas_y * ((ngroups + ngrp - 1) / ngrp) < 2LL * sm_count) --ngrp;
    a->ngrp = ngrp;
}

// k_poly blocks per CTA: from `start` down to what shared memory holds (their parked spectra) and what keeps the grid at
// two CTAs per SM, balanced -- the per-CTA tables are built once and the inverse rounds fill up (measured on C1, 7 blocks
// per stream: 1.93 / 1.74 / 1.66 ms with 1 / 2 / 7 blocks per CTA)
template <typename T> int poly_nbpc(int K, int Q, int G, int S, int n_blocks, int start, int sm_count) {
    int nbpc = start;
    while (nbpc > 1 && rr::poly_smem_bytes<T>(K, Q, G, nbpc) > (size_t)200 * 1024) --nbpc;
    while (nbpc > 1 && (long long)S * ((n_blocks + nbpc - 1) / nbpc) < 2LL * sm_count) --nbpc;
    const int nsb = (n_blocks + nbpc - 1) / nbpc;
    return (n_blocks + nsb - 1) / nsb;
}

// the front ends' rows row_first .. row_first + n_rows - 1 of every stream to u, and the part of the Filter's next
// history that rows up to push offset cover_hi reach
rr::FrontArgs front_args(const PolyPart& p, const DevBuf& acoef, long long row_first, long long n_rows, void* u, long long u_stride,
                         long long cover_hi) {
    rr::FrontArgs fa{};
    fa.in = p.io.in;
    fa.in_stride = p.io.in_stride;
    fa.len = p.len;
    fa.hist2 = p.f.hist2[p.f.hist_cur].p;
    fa.n = p.n;
    fa.nco = p.nco;
    fa.acoef = (const float*)acoef.p;
    fa.P = (int)p.P;
    fa.J0 = p.J0;
    fa.row_first = row_first;
    fa.n_rows = (int)n_rows;
    fa.u = u;
    fa.u_stride = u_stride;
    fa.hist_staged = next_history(p, row_first * p.P - p.J0, cover_hi, &fa) && p.len < 4 * p.n;  // measured: pays off up to 3 chunks per push
    return fa;
}

// the k_poly / k_poly2 arguments of the polyphase chain on the input itself
template <typename T> rr::PolyArgs<T> input_poly_args(const PolyPart& p) {
    rr::PolyArgs<T> a{};
    a.in = p.io.in;
    a.in_stride = p.io.in_stride;
    a.len = p.len;
    a.hist2 = p.f.hist2[p.f.hist_cur].p;
    a.n = p.n;
    a.nco = p.nco;
    a.gtab = p.ds.gtab.p;
    a.twK = p.ds.twK.p;
    a.P = p.P;
    a.Q = p.Q;
    a.Lmax = p.ds.poly_Lmax;
    a.V = p.ds.poly_V;
    a.J0 = p.J0;
    a.m0 = p.m0;
    a.m_lo = p.m_lo;
    a.m_hi = p.m_hi;
    a.I_lo = p.I_lo;
    a.out = p.obase;
    a.out_stride = p.ostride;
    return a;
}

// The routes, tried in this order by run_filter_down.  Each checks its preconditions first; when they hold it launches
// its kernels and names itself in *route, else it leaves *route unset and the next route is tried.

// k_fused: front end + low-rate part in one persistent kernel (u stays in shared memory).  Steady state only: the whole
// push is polyphase, the previous push left its last Lmax rows of u behind, and there are enough streams to give every
// SM whole streams; everything else takes k_front + k_poly2.
int route_fused(const PolyPart& p, const char** route) {
    rr_chain* c = p.c;
    Stage& ds = p.ds;
    const long long n_out = p.m_hi - p.m_lo + 1;
    if (!(ds.poly2_valid && ds.front_valid && ds.fused_valid && c->allow_fused && p.tma_ok && p.kept && ds.ucache_ptr && p.Q == 1 &&
          p.m0 == 0 && p.J0 >= 0 && p.J0 < p.P && c->S >= c->fused_min_streams && n_out >= c->fused_min_rows && p.len >= 33 * p.P))
        return RR_OK;
    constexpr int RK = 10;
    const long long Lh = ds.poly_Lmax;
    DevBuf& kb = ds.ukeep[ds.ukeep_cur];
    RR_TRY(kb.ensure((size_t)c->S * (size_t)Lh * RK * 2 * sizeof(float)));
    rr::FusedArgs fu{};
    fu.in = p.io.in;
    fu.in_stride = p.io.in_stride;
    fu.len = p.len;
    fu.hist2 = p.f.hist2[p.f.hist_cur].p;
    fu.n = p.n;
    fu.nco = p.nco;
    fu.P = (int)p.P;
    fu.coef_slot = ds.fused_slot;
    fu.J0 = p.J0;
    fu.n_out = (int)n_out;
    fu.Lmax = (int)Lh;
    fu.V = ds.poly2_V;
    fu.ukeep_in = ds.ucache_ptr;
    fu.ukeep_in_stride = ds.ucache_stride;
    fu.ukeep_out = kb.p;
    fu.ukeep_out_stride = Lh * RK;
    fu.gtab = ds.gtab3.p;
    fu.twK = ds.poly2_tw_own ? ds.twK2.p : ds.twK.p;
    fu.out = p.obase;
    fu.out_stride = p.ostride;
    direct_split(p, &fu);
    // the rows cover push offsets [-J0, m_hi*P - J0)
    next_history(p, -p.J0, p.m_hi * p.P - p.J0, &fu);
    RR_TIMED_LAUNCH(c, "k_fused", 1, rr::launch_fused(c->S, fu, p.io.shared, c->ctx->sm_count, c->stream));
    ds.ucache_valid = true;
    ds.ucache_rows = n_out + Lh;
    ds.ucache_ptr = kb.p;
    ds.ucache_stride = Lh * RK;
    ds.ukeep_cur ^= 1;
    *route = "fused[filter+down]";
    return RR_OK;
}

// k_front + k_poly2 (Q == 1, the filter factors to rank 10): u rows [m_lo-1-Lmax, m_hi-1] of every stream, then the
// low-rate part on u as a stream of RK branches whose first output (virtual index Lmax+1) is output m_lo
int route_front_poly2(const PolyPart& p, const char** route) {
    rr_chain* c = p.c;
    Stage& ds = p.ds;
    if (!(ds.poly2_valid && ds.front_valid && p.tma_ok)) return RR_OK;
    constexpr int RK = 10;
    const int S = c->S;
    const long long Lh = ds.poly_Lmax;
    const long long n_out = p.m_hi - p.m_lo + 1;
    const long long n_rows = n_out + Lh;
    if (n_rows >= (1LL << 27)) return RR_OK;
    // every stream's rows are followed by one transform length of zero rows, so that the low-rate part
    // reads whole tiles by TMA up to and including its last block (no edge path, no shifted block)
    // (rows beyond n_rows only feed outputs that are not stored; the stride is rounded so that pushes whose
    // output count differs by a few keep the layout, and what an earlier push left there is that stream's own)
    const long long pad_rows = 512;
    const long long u_stride = (((n_rows + 127) / 128 * 128 + pad_rows) * RK + 1) / 2 * 2;
    // short pushes (one block per stream): the low-rate part takes runs of sab_nb streams as the blocks of
    // one "stream", so that an inverse round serves several streams (PolyArgs::sab_*)
    const int n_blocks1 = (int)((n_out - 1) / ds.poly2_V + 1);
    const int halves_total = 2 * c->ctx->sm_count;
    const int sab_run = (c->allow_sab && n_blocks1 <= 3 && S > halves_total) ? (S + halves_total - 1) / halves_total : 0;  // streams
    const int sab_nb = sab_run * n_blocks1;  // blocks of a run
    const size_t S_alloc = sab_run ? (size_t)((S + sab_run - 1) / sab_run) * sab_run : (size_t)S;
    const size_t ubytes = S_alloc * (size_t)u_stride * 2 * sizeof(float);
    DevBuf& ub = ds.ubuf[ds.ubuf_cur];
    if (ub.bytes < ubytes || ds.ubuf_stride[ds.ubuf_cur] != u_stride) {
        // a new layout: the pad rows must read as zeros (they only ever feed outputs that are not stored,
        // but a NaN there would spread through the transform)
        RR_TRY(ub.ensure(ubytes));
        RR_CUDA(cudaMemsetAsync(ub.p, 0, ubytes, c->stream));
        ds.ubuf_stride[ds.ubuf_cur] = u_stride;
    }
    // history rows: kept from the previous push when it went through here too (k_front moves them over itself), else
    // recomputed from hist2
    const bool cached = p.kept && ds.ucache_rows >= Lh && n_out > 0;
    rr::FrontArgs fa = front_args(p, ds.acoef, p.m_lo - 1 - (cached ? 0 : Lh), cached ? n_out : n_rows,
                                  (char*)ub.p + (cached ? (size_t)Lh * RK * 2 * sizeof(float) : 0), u_stride, p.m_hi * p.P - p.J0);
    if (cached) {
        fa.kept_src = ds.ucache_ptr;
        fa.kept_stride = ds.ucache_stride;
        fa.kept_rows = (int)Lh;
    }
    RR_TIMED_LAUNCH(c, "k_front", 1, rr::launch_front(RK, S, fa, p.io.shared, c->ctx->sm_count, c->stream));
    rr::PolyArgs<float> b{};
    b.in = ub.p;
    b.in_stride = u_stride;
    b.len = (n_rows + pad_rows) * RK;
    b.hist2 = ub.p;
    b.n = 0;
    b.nco = nullptr;
    b.gtab = ds.gtab3.p;
    b.twK = ds.poly2_tw_own ? ds.twK2.p : ds.twK.p;
    b.P = RK;
    b.Q = 1;
    b.Lmax = ds.poly_Lmax;
    b.V = ds.poly2_V;
    b.J0 = 0;
    b.m0 = ds.poly_Lmax;
    b.m_lo = ds.poly_Lmax + 1;
    b.m_hi = ds.poly_Lmax + n_out;
    b.I_lo = b.m_lo;
    b.n_blocks = (int)((b.m_hi - b.I_lo) / b.V + 1);
    poly2_grid(&b, RK, S, c->ctx->sm_count);
    b.out = p.obase;
    b.out_stride = p.ostride;
    int S2 = S;  // streams of the low-rate launch
    if (sab_nb) {
        int nb2 = std::min(RK, sab_nb);
        while (nb2 > 1 && rr::poly2_smem_bytes(RK, nb2) > (size_t)226 * 1024) --nb2;
        const int groups2 = (sab_nb + nb2 - 1) / nb2;
        b.n_blocks = sab_nb;
        b.nbpc = (sab_nb + groups2 - 1) / groups2;
        b.ngrp = groups2;  // a half takes all groups of its run of streams
        b.sab_blocks = sab_nb;
        b.sab_rb = n_blocks1;
        b.sab_streams = S;
        b.sab_in_step = u_stride;
        b.in_stride = (long long)sab_run * u_stride;
        b.len = (long long)sab_run * u_stride;
        S2 = (S + sab_run - 1) / sab_run;
    }
    if (p.whole) direct_split(p, &b);
    if (sab_nb) {
        b.sab_out_step = b.out_stride;
        b.sab_out2_step = b.out2_stride;
        b.out_stride *= sab_run;
        b.out2_stride *= sab_run;
    }
    RR_TIMED_LAUNCH(c, "k_poly2", 1, rr::launch_poly2(RK, S2, b, false, c->ctx->sm_count, c->stream));
    ds.ucache_valid = true;
    ds.ucache_rows = n_rows;
    // the last Lmax rows of [history rows | new rows] of this push
    ds.ucache_ptr = (const char*)ub.p + (size_t)(n_rows - Lh) * RK * 2 * sizeof(float);
    ds.ucache_stride = u_stride;
    ds.ubuf_cur ^= 1;
    *route = "front+poly2[filter+down]";
    return RR_OK;
}

// k_front / k_front_wide + k_poly (Q > 1): u rows [I_lo-1-Lmax, I_hi] (tap l = -1 of the phases q > 0 reads row I),
// then k_poly on u with the Q phase tables.  Output m = Q*I + q keeps its index: block 0's window starts at u row 0,
// which is row I_lo-1-Lmax of the stream (PolyArgs::J0 in units of u samples).  No rows are kept between pushes (the
// last row of a push is cut off by its end).
int route_front_q(const PolyPart& p, const char** route) {
    rr_chain* c = p.c;
    Stage& ds = p.ds;
    if (!(ds.frontq_valid && (p.tma_ok || ds.frontq_wide) && p.Q > 1)) return RR_OK;
    const int S = c->S;
    const int RQ = ds.frontq_cols;
    constexpr int GQ = 8;
    const long long Lh = ds.poly_Lmax;
    const long long row_first = p.I_lo - 1 - Lh;
    const long long n_rows = p.I_hi - p.I_lo + 2 + Lh;
    const long long u_stride = n_rows * RQ;
    if (n_rows * p.P >= (1LL << 31)) return RR_OK;
    DevBuf& ub = ds.ubuf[0];
    RR_TRY(ub.ensure((size_t)S * (size_t)u_stride * 2 * sizeof(float)));
    ds.ubuf_stride[0] = -1;
    // the rows cover push offsets up to (I_hi+1)*P - J0, cut off at the end of the push
    const rr::FrontArgs fa = front_args(p, ds.acoef_q, row_first, n_rows, ub.p, u_stride, std::min<long long>((p.I_hi + 1) * p.P - p.J0, p.len));
    if (ds.frontq_wide) RR_TIMED_LAUNCH(c, "k_front_wide", 1, rr::launch_front_wide(RQ, S, fa, c->stream));
    else RR_TIMED_LAUNCH(c, "k_front", 1, rr::launch_front(RQ, S, fa, p.io.shared, c->ctx->sm_count, c->stream));
    rr::PolyArgs<float> b{};
    b.in = ub.p;
    b.in_stride = u_stride;
    b.len = n_rows * RQ;
    b.hist2 = ub.p;
    b.n = 0;
    b.nco = nullptr;
    b.gtab = ds.gtab_q.p;
    b.twK = ds.twK.p;
    b.P = RQ;
    b.Q = p.Q;
    b.Lmax = (int)Lh;
    b.V = ds.poly_V;
    b.J0 = row_first * RQ;
    b.m0 = p.m0;
    b.m_lo = p.m_lo;
    b.m_hi = p.m_hi;
    b.I_lo = p.I_lo;
    b.n_blocks = (int)((p.I_hi - p.I_lo) / b.V + 1);
    b.nbpc = poly_nbpc<float>(ds.poly_K, (int)p.Q, GQ, S, b.n_blocks, b.n_blocks, c->ctx->sm_count);
    b.out = p.obase;
    b.out_stride = p.ostride;
    RR_TIMED_LAUNCH(c, "k_poly(u)", 1, rr::launch_poly<float>(ds.poly_K, (int)p.Q, GQ, S, b, c->stream));
    *route = "front+poly[filter+down]";
    return RR_OK;
}

// k_poly2 on all P branches of the input (Q == 1, a filter that does not factor to rank 10)
int route_poly2(const PolyPart& p, const char** route) {
    rr_chain* c = p.c;
    Stage& ds = p.ds;
    if (!(ds.poly2_valid && p.tma_ok)) return RR_OK;
    rr::PolyArgs<float> a = input_poly_args<float>(p);
    a.gtab = ds.gtab2.p;
    if (ds.poly2_tw_own) a.twK = ds.twK2.p;
    a.V = ds.poly2_V;
    a.n_blocks = (int)((p.I_hi - p.I_lo) / a.V + 1);
    poly2_grid(&a, ds.poly2_G, c->S, c->ctx->sm_count);
    RR_TIMED_LAUNCH(c, "k_poly2", 1, rr::launch_poly2(ds.poly2_G, c->S, a, p.io.shared, c->ctx->sm_count, c->stream));
    *route = "poly2[filter+down]";
    return RR_OK;
}

// k_poly: the generic polyphase kernel (f32 and f64, any Q <= 4); blocks per CTA start at one round of inverse
// transforms (G jobs)
template <typename T> int route_poly(const PolyPart& p, const char** route) {
    rr_chain* c = p.c;
    Stage& ds = p.ds;
    rr::PolyArgs<T> a = input_poly_args<T>(p);
    a.n_blocks = (int)((p.I_hi - p.I_lo) / a.V + 1);
    a.nbpc = poly_nbpc<T>(ds.poly_K, (int)p.Q, ds.poly_G, c->S, a.n_blocks, std::max(1, ds.poly_G / (int)p.Q), c->ctx->sm_count);
    RR_TIMED_LAUNCH(c, "k_poly", 1, rr::launch_poly<T>(ds.poly_K, (int)p.Q, ds.poly_G, c->S, a, c->stream));
    *route = "poly[filter+down]";
    return RR_OK;
}

template <typename T>
int run_filter_down(rr_chain* c, Stage& f, Stage& ds, const FilterIo& io, const StageAct& fa, const StageAct& da, std::string* plan,
                    DirectOut* direct = nullptr) {
    const size_t n = io.n;
    const int S = c->S;
    cudaStream_t st = c->stream;
    const int L = ds.h.r_L;
    void* obase = (char*)ds.obuf[ds.obuf_cur].p + da.pending_before * 2 * sizeof(T);
    const long long ostride = (long long)ds.obuf_cap;

    const bool rational = !ds.h.r_indexed && is_pow2(n);  // the fused polyphase / overlap-save+FIR kernels need in/out = P/Q and a power-of-two chunk
    if (c->allow_poly && rational) RR_TRY(poly_prepare<T>(c, f, ds));
    // the kept u rows stay usable only from one front-end push to the very next one
    const bool was_ucache_valid = ds.ucache_valid;
    ds.ucache_valid = false;
    // chunks the stateful path must take: those whose outputs still depend on pre-segment state
    size_t ca = io.n_chunks;
    if (c->allow_poly && rational && ds.poly_valid) {
        const size_t need = (size_t)(2 - std::min(2, fa.seg_before));
        ca = std::min(need, io.n_chunks);
    }
    const size_t fih = fa.first_is_history ? 1 : 0;

    // ---- stateful part: chunks [0, ca) ------------------------------------------
    long long j0 = da.j0, m0 = da.m0;  // decimator counters at the start of the part being processed
    if (ca > fih) {
        const long long zlen = (long long)((ca - fih) * n);
        if (ds.h.r_indexed) {
            // rates that are not integer valued: Filter output to scratch, then the FIR at the firing instants of the
            // reference's f64 recurrence
            RR_TRY(f.ztmp.ensure((size_t)S * (size_t)zlen * 2 * sizeof(T)));
            RR_TRY(run_os<T>(c, f, io, ca, fih != 0, f.ztmp.p, zlen));
            RR_TRY(downsample_indexed<T>(c, ds, da, f.ztmp.p, zlen, zlen, obase, ostride));
            *plan += "os|downsample(indexed)";
            return RR_OK;
        }
        const long long tot = floordiv128(j0 + zlen, ds.h.Q, ds.h.P);
        const long long n_out = tot - m0;
        if (rational && rr::chain_os_supported<T>((int)n, 1, L)) {
            rr::ChainOsArgs<T> a{};
            a.in = io.in;
            a.in_stride = io.in_stride;
            a.n_chunks = (int)ca;
            a.first_is_history = (int)fih;
            a.emit = 1;
            a.hist_in = (const char*)f.hist2[f.hist_cur].p + n * 2 * sizeof(T);
            a.hist_stride = (long long)(2 * n);
            a.hist_out = nullptr;
            a.hperm = f.hperm.p;
            a.twN = f.tw.p;
            a.nco = io.nco ? (const rr::NcoStream*)io.nco->nco_d.p : nullptr;
            a.nco_offset = 0;
            a.out = obase;
            a.out_stride = ostride;
            a.ir = (const T*)ds.ir.p;
            a.L = L;
            a.ztail_in = ds.tail[ds.tail_cur].p;
            a.ztail_out = ds.tail[ds.tail_cur ^ 1].p;
            a.rate.P = ds.h.P;
            a.rate.Q = ds.h.Q;
            a.rate.j0 = j0;
            a.rate.m0 = m0;
            RR_TIMED_LAUNCH(c, "k_chain_os<epi=down>", 1, rr::launch_chain_os<T>((int)n, 1, S, 1, a, st));
            ds.tail_cur ^= 1;
            *plan += "fused_os[filter+down]";
        } else {
            RR_TRY(f.ztmp.ensure((size_t)S * (size_t)zlen * 2 * sizeof(T)));
            RR_TRY(run_os<T>(c, f, io, ca, fih != 0, f.ztmp.p, zlen));
            rr::RateState rs;
            rs.P = ds.h.P;
            rs.Q = ds.h.Q;
            rs.j0 = j0;
            rs.m0 = m0;
            RR_LAUNCH(2, rr::launch_downsample<T>(f.ztmp.p, zlen, zlen, ds.tail[ds.tail_cur].p, ds.tail[ds.tail_cur ^ 1].p, (const T*)ds.ir.p,
                                                  L, rs, n_out, obase, ostride, S, st));
            ds.tail_cur ^= 1;
            *plan += !is_pow2(n) ? "padded_os[filter]|downsample" : (rr::chain_os_supported<T>((int)n, 0, 0) ? "fused_os[filter]|downsample" : "big_os|downsample");
        }
        obase = (char*)obase + (size_t)n_out * 2 * sizeof(T);
        j0 = (j0 + zlen) % ds.h.P;
        m0 = floordiv128(j0, ds.h.Q, ds.h.P);
    }
    if (ca == io.n_chunks) return RR_OK;

    // ---- polyphase part: chunks [ca, n_chunks) ----------------------------------------
    const long long P = ds.h.P, Q = ds.h.Q, len = (long long)(io.n_chunks * n);
    const long long m_lo = m0 + 1, m_hi = floordiv128(j0 + (long long)((io.n_chunks - ca) * n), Q, P);
    const bool whole = ca == 0;
    const PolyPart p{c, f, ds, io, da, direct, P, Q, j0 - (long long)(ca * n), m0, m_lo, m_hi, m_lo / Q, m_hi / Q, len, (long long)n,
                     io.nco ? (const rr::NcoStream*)io.nco->nco_d.p : nullptr, obase, ostride,
                     rr::tma_input_ok(io.in, io.in_stride, len, S, io.shared), whole, whole && was_ucache_valid && c->allow_ucache};
    const char* route = nullptr;
    if (m_hi < m_lo) route = "poly[filter+down]";  // no output fires in this part
    if constexpr (std::is_same<T, float>::value) {
        if (!route) RR_TRY(route_fused(p, &route));
        if (!route) RR_TRY(route_front_poly2(p, &route));
        if (!route) RR_TRY(route_front_q(p, &route));
        if (!route) RR_TRY(route_poly2(p, &route));
    }
    if (!route) RR_TRY(route_poly<T>(p, &route));
    ds.ztail_stale = true;
    if (!plan->empty() && plan->back() != '+' && plan->back() != '|' && ca > 0) *plan += "|";
    *plan += route;
    return RR_OK;
}

// The summed push's fused route (k_synth): the chain ends Upsampler -> FreqShifter, the Upsampler takes
// k_upsample_phase's integer-factor form in this push (`up`: its state after the push's dry run), and the push emits.
bool synth_route(const rr_chain* c, const std::vector<StageHost>& hs, const Shape& out) {
    const int ns = (int)c->st.size();
    if (ns < 2 || c->st[ns - 2].d.kind != RR_STAGE_UPSAMPLE || c->st[ns - 1].d.kind != RR_STAGE_FREQSHIFT || out.len() == 0) return false;
    const StageHost& up = hs[ns - 2];
    return up.r_valid && !up.r_indexed && rr::upsample_phase_supported(rr::RateState{up.P, up.Q, 0, 0}, up.r_L, (long long)out.len());
}

// shared: every stream reads the row at dev_in (in_stride is 0).  The stride travels with the input view, so every
// stage that reads the push's input sees it; the TMA launchers take their shared-row form on a zero stride.
// summed: dev_out is ONE row (out_stride unused) that receives the sum over streams of the per-stream outputs
// (rr_chain_push_summed).  Off the k_synth route the stages write the per-stream outputs into c->sum_rows exactly as a
// per-stream push writes the caller's buffer, and k_stream_sum adds them into the row.
template <typename T>
int run_push(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in, size_t in_stride, bool shared,
             bool summed, void* dev_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_rate) {
    const int S = c->S;
    const int ns = (int)c->st.size();
    cudaStream_t st = c->stream;
    Shape in;
    in.chunk_len = chunk_len;
    in.n_chunks = n_chunks;
    in.rate = sample_rate;
    if (shared) in_stride = 0;
    else if (chunk_len * n_chunks > in_stride && S > 1) return fail(RR_ERR_INVALID, "in_stride smaller than the pushed samples");

    // ---- dry run: output shape + capacity before anything is touched -------
    bool synth = false;
    void* const row_out = dev_out;  // summed: the caller's row
    {
        Shape sh;
        std::vector<StageHost> hs;
        RR_TRY(dry_shape(c, in, &sh, &hs));
        if (sh.len() > out_capacity) return fail(RR_ERR_CAPACITY, "output buffer too small for this push");
        if (!summed && sh.len() > out_stride && S > 1) return fail(RR_ERR_INVALID, "out_stride smaller than the produced samples");
        if (summed && sh.len() > 0 && !dev_out) return fail(RR_ERR_INVALID, "rr_chain_push_summed_device: dev_out is null");
        if (summed) synth = synth_route(c, hs, sh);
        if (summed && !synth && sh.len() > 0) {
            RR_TRY(c->sum_rows.ensure((size_t)S * sh.len() * c->esz));
            dev_out = c->sum_rows.p;
            out_stride = sh.len();
        }
    }

    c->push_mutated = true;
    std::string plan;
    View cur;
    cur.p = dev_in;
    cur.stride = (long long)in_stride;
    cur.sh = in;
    Stage* pending_nco = nullptr;  // FreqShifter deferred into the next Filter's load stage

    for (int i = 0; i < ns; ++i) {
        Stage& s = c->st[i];
        const bool last = (i == ns - 1);
        // the Filter needs its pre-redesign state once more when a polyphase push left the decimator tail stale
        if (s.d.kind == RR_STAGE_FILTER && !last && c->st[i + 1].d.kind == RR_STAGE_DOWNSAMPLE && c->st[i + 1].ztail_stale &&
            cur.sh.n_chunks > 0) {
            StageHost probe = s.h;
            StageAct pa;
            RR_TRY(advance_stage(s.d, probe, cur.sh, &pa));
            StageHost dprobe = c->st[i + 1].h;
            StageAct dpa;
            int r = advance_stage(c->st[i + 1].d, dprobe, pa.out, &dpa);
            const bool ds_redesign = (r == RR_OK) && dpa.redesign;
            if (ds_redesign) c->st[i + 1].ztail_stale = false;  // the ring restarts from zero anyway
            else if (pa.redesign || pa.first_is_history || !c->allow_poly) RR_TRY(regen_ztail<T>(c, s, c->st[i + 1]));
        }
        StageAct a;
        RR_TRY(advance_stage(s.d, s.h, cur.sh, &a));
        if (a.lost) {  // SamplesLost travels ahead of the samples (chunks.rs:71-79)
            ++c->samples_lost;
            bool intr = true;
            for (int j = i + 1; j < ns; ++j) c->samples_lost += (uint64_t)stage_event(c->st[j].d, c->st[j].h, &intr);
        }
        if (!a.active) {
            cur.sh = a.out;
            continue;
        }
        const long long len = (long long)cur.sh.len();
        if (!plan.empty() && plan.back() != '+') plan += "|";
        switch (s.d.kind) {
            case RR_STAGE_FREQSHIFT: {
                RR_TRY(nco_refresh<T>(c, s, cur.sh.rate, a.nco_recalc));
                const size_t n = cur.sh.chunk_len;
                const bool fuse = !last && c->st[i + 1].d.kind == RR_STAGE_FILTER && n >= 32 && (n & (n - 1)) == 0 &&
                                  (rr::chain_os_supported<T>((int)n, 0, 0) || rr::big_os_supported<T>((int)n));
                if (fuse) {
                    pending_nco = &s;
                    plan += "nco+";
                } else {
                    Dest d;
                    RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, (size_t)len, &d));
                    RR_TIMED_LAUNCH(c, "k_freqshift", 1, rr::launch_freqshift<T>(cur.p, cur.stride, d.p, d.stride, len, S, (const rr::NcoStream*)s.nco_d.p, 0, st));
                    RR_LAUNCH(1, rr::launch_nco_advance((rr::NcoStream*)s.nco_d.p, S, len, st));
                    nco_host_advance(s, len);
                    cur.p = d.p;
                    cur.stride = d.stride;
                    plan += "freqshift";
                }
                cur.sh = a.out;
                break;
            }
            case RR_STAGE_GAIN: {
                Dest d;
                RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, (size_t)len, &d));
                RR_TIMED_LAUNCH(c, "k_gain", 1, rr::launch_gain<T>(cur.p, cur.stride, d.p, d.stride, len, S, s.d.gain, st));
                cur.p = d.p;
                cur.stride = d.stride;
                cur.sh = a.out;
                plan += "gain";
                break;
            }
            case RR_STAGE_FOURIER: {
                const size_t n = cur.sh.chunk_len;
                if (!rr::fourier_fft_supported<T>((int)n) && n > (size_t)rr::kFourierDirectMax)
                    return fail(RR_ERR_UNSUPPORTED, "Fourier: chunk lengths outside the FFT plans are limited to 4096 samples");
                if (s.fwin_n != n) {
                    // analysis.rs:86-103: window sampled at the bin centres, scaled to unit mean power, rounded to Flt
                    rr::WindowFn w = make_window(s.d.window_kind, s.d.window_beta, s.d.window_fn, s.d.window_user);
                    std::vector<double> wv(n);
                    double energy = 0.0;
                    for (size_t k = 0; k < n; ++k) {
                        wv[k] = w(2.0 * ((double)k + 0.5) / (double)n - 1.0);
                        energy += wv[k] * wv[k];
                    }
                    const double scale = std::sqrt((double)n / energy);
                    for (auto& v : wv) v *= scale;
                    RR_TRY(upload_real<T>(s.fwin, wv, st));
                    if (rr::fourier_fft_supported<T>((int)n)) {
                        std::vector<std::complex<double>> tw;
                        rr::make_twiddles(n, &tw);
                        RR_TRY(upload_complex<T>(s.ftw, tw, st));
                    }
                    s.fwin_n = n;
                }
                Dest d;
                RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, (size_t)len, &d));
                RR_TIMED_LAUNCH(c, "k_fourier", 1, rr::launch_fourier<T>((int)n, cur.p, cur.stride, d.p, d.stride, (int)cur.sh.n_chunks, S, (const T*)s.fwin.p,
                                                   s.ftw.p, s.d.center_dc ? (int)(n / 2) : 0, st));
                cur.p = d.p;
                cur.stride = d.stride;
                cur.sh = a.out;
                plan += "fourier";
                break;
            }
            case RR_STAGE_FMMOD: {
                Dest d;
                RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, (size_t)len, &d));
                RR_TRY(s.fm_phase.ensure((size_t)S * sizeof(T), true, st));
                const double factor = s.d.deviation / cur.sh.rate * 6.283185307179586476925286766559;  // modulation.rs:44
                RR_TIMED_LAUNCH(c, "k_fmmod", 1, rr::launch_fmmod<T>(cur.p, cur.stride, d.p, d.stride, len, S, s.fm_phase.p, factor, c->ctx->sm_count, st));
                cur.p = d.p;
                cur.stride = d.stride;
                cur.sh = a.out;
                plan += "fmmod";
                break;
            }
            case RR_STAGE_RECHUNK: {
                // the sequence [partial chunk | pushed samples]: whole chunks go on, the rest is kept (chunks.rs:100-164)
                const size_t p0 = a.pending_before, emit = a.out.len(), n_new = a.n_new;
                const size_t from_p = std::min(p0, emit), from_in = emit - from_p;
                RR_TRY(obuf_reserve<T>(c, s, std::max<size_t>((size_t)s.d.output_chunk_len, p0 + (emit ? 0 : n_new)), p0));
                const long long ocap = (long long)s.obuf_cap;
                const char* pend = (const char*)s.obuf[s.obuf_cur].p;
                const char* inp = (const char*)cur.p;
                const long long in_str = cur.stride;
                const size_t esz = 2 * sizeof(T);
                if (emit == 0) {
                    RR_LAUNCH(1, rr::launch_copy2d<T>(inp, in_str, (char*)s.obuf[s.obuf_cur].p + p0 * esz, ocap, (long long)n_new, S, st));
                    cur.sh = a.out;
                    plan += "rechunk(hold)";
                    break;
                }
                char* other = (char*)s.obuf[s.obuf_cur ^ 1].p;
                if (p0 == 0 && !last) {
                    plan += "rechunk(view)";  // the pushed buffer itself, seen with the new chunk length
                } else {
                    Dest d;
                    RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, emit, &d));
                    if (from_p) RR_LAUNCH(1, rr::launch_copy2d<T>(pend, ocap, d.p, d.stride, (long long)from_p, S, st));
                    if (from_in) RR_LAUNCH(1, rr::launch_copy2d<T>(inp, in_str, (char*)d.p + from_p * esz, d.stride, (long long)from_in, S, st));
                    cur.p = d.p;
                    cur.stride = d.stride;
                    plan += "rechunk";
                }
                if (p0 > from_p) RR_LAUNCH(1, rr::launch_copy2d<T>(pend + from_p * esz, ocap, other, ocap, (long long)(p0 - from_p), S, st));
                if (n_new > from_in)
                    RR_LAUNCH(1, rr::launch_copy2d<T>(inp + from_in * esz, in_str, other + (p0 - from_p) * esz, ocap, (long long)(n_new - from_in), S, st));
                s.obuf_cur ^= 1;
                cur.sh = a.out;
                break;
            }
            case RR_STAGE_OVERLAP: {
                const size_t k = (size_t)s.d.chunk_count, n = cur.sh.chunk_len, h0 = a.pending_before;
                const size_t tot = h0 + cur.sh.n_chunks, n_out = a.out.n_chunks, h1 = std::min(k - 1, tot);
                if ((k - 1) * n > s.tail_cap || (k > 1 && (!s.tail[0].p || !s.tail[1].p))) {
                    // only reached with an empty history (the history's chunk length is fixed while it holds chunks)
                    RR_TRY(s.tail[0].ensure((size_t)S * (k - 1) * n * 2 * sizeof(T)));
                    RR_TRY(s.tail[1].ensure((size_t)S * (k - 1) * n * 2 * sizeof(T)));
                    s.tail_cap = (k - 1) * n;
                }
                const void* hist = s.tail[s.tail_cur].p;
                const void* inp = cur.p;
                const long long in_str = cur.stride;
                if (n_out > 0) {
                    Dest d;
                    RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, a.out.len(), &d));
                    RR_LAUNCH(1, rr::launch_overlap<T>(hist, (long long)s.tail_cap, (long long)(h0 * n), inp, in_str, d.p, d.stride, (long long)n_out,
                                                       (long long)(k * n), (long long)n, 0, S, st));
                    cur.p = d.p;
                    cur.stride = d.stride;
                }
                if (h1 > 0) {
                    RR_LAUNCH(1, rr::launch_overlap<T>(hist, (long long)s.tail_cap, (long long)(h0 * n), inp, in_str, s.tail[s.tail_cur ^ 1].p,
                                                       (long long)s.tail_cap, 1, (long long)(h1 * n), 0, (long long)((tot - h1) * n), S, st));
                    s.tail_cur ^= 1;
                }
                cur.sh = a.out;
                plan += "overlap";
                break;
            }
            case RR_STAGE_FMDEMOD: {
                Dest d;
                RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, (size_t)len, &d));
                RR_TRY(s.fm_prev.ensure((size_t)S * 2 * sizeof(T), true, st));
                RR_TRY(s.fm_last.ensure((size_t)S * 2 * sizeof(T), true, st));
                const double factor = cur.sh.rate / s.d.deviation / 6.283185307179586476925286766559;  // modulation.rs:116
                RR_TIMED_LAUNCH(c, "k_fmdemod", 2, rr::launch_fmdemod<T>(cur.p, cur.stride, d.p, d.stride, len, S, s.fm_prev.p, s.fm_last.p,
                                                   a.first_is_history ? 0 : 1, factor, st));
                cur.p = d.p;
                cur.stride = d.stride;
                cur.sh = a.out;
                plan += "fmdemod";
                break;
            }
            case RR_STAGE_FILTER: {
                const size_t n = cur.sh.chunk_len;
                if (a.redesign) {
                    RR_TRY(filter_redesign<T>(c, s, cur.sh.rate, n));
                    if (!last && c->st[i + 1].d.kind == RR_STAGE_DOWNSAMPLE) {
                        c->st[i + 1].poly_valid = false;
                        c->st[i + 1].poly_tried = false;
                    }
                }
                FilterIo io;
                io.in = cur.p;
                io.shared = shared && S > 1 && cur.p == dev_in;  // still the pushed row (a Rechunker view keeps it)
                io.in_stride = cur.stride;
                io.n = n;
                io.n_chunks = cur.sh.n_chunks;
                io.nco = pending_nco;
                pending_nco = nullptr;
                Stage* ds = (!last && c->st[i + 1].d.kind == RR_STAGE_DOWNSAMPLE) ? &c->st[i + 1] : nullptr;
                bool took_ds = false;
                if (ds && a.out.n_chunks > 0) {
                    // Filter -> Downsampler handled together (fused kernels)
                    StageAct da;
                    RR_TRY(advance_stage(ds->d, ds->h, a.out, &da));
                    if (da.redesign) {
                        RR_TRY(resampler_redesign<T>(c, *ds, a.out.rate));
                    }
                    RR_TRY(obuf_reserve<T>(c, *ds, da.pending_before + da.n_new, da.pending_before));
                    const bool ds_last = (i + 1 == ns - 1);
                    DirectOut direct;
                    if (ds_last) {
                        direct.user_out = dev_out;
                        direct.user_stride = (long long)out_stride;
                    }
                    RR_TRY(run_filter_down<T>(c, s, *ds, io, a, da, &plan, &direct));
                    RR_TRY(resampler_emit<T>(c, *ds, da, ds_last, dev_out, (long long)out_stride, &cur, direct.done));
                    took_ds = true;
                } else {
                    if (ds) ds->ucache_valid = false;
                    Dest d;
                    RR_TRY(pick_dest<T>(c, s, last, dev_out, (long long)out_stride, a.out.len(), &d));
                    RR_TRY(run_os<T>(c, s, io, io.n_chunks, a.first_is_history, d.p, d.stride));
                    cur.p = d.p;
                    cur.stride = d.stride;
                    cur.sh = a.out;
                    plan += !is_pow2(n) ? "padded_os[filter]" : (rr::chain_os_supported<T>((int)n, 0, 0) ? "fused_os[filter]" : "big_os");
                }
                // new history: the last two mixed chunks (filters.rs:260 keeps one; the polyphase path needs two)
                {
                    const void* hin = s.hist2[s.hist_cur].p;
                    void* hout = s.hist2[s.hist_cur ^ 1].p;
                    const rr::NcoStream* ncop = io.nco ? (const rr::NcoStream*)io.nco->nco_d.p : nullptr;
                    if (s.hist_fused_jlo > 0) {
                        // k_front wrote [jfirst, jlo): the old history in front of it and the samples behind its last row remain
                        if (s.hist_fused_jfirst > 0)
                            RR_TIMED_LAUNCH(c, "k_hist2_update", 1, rr::launch_hist2_update<T>(io.in, io.in_stride, len, hin, hout, (long long)n, ncop, S,
                                                                                                st, 0, s.hist_fused_jfirst));
                        if (s.hist_fused_jlo < (long long)(2 * n))
                            RR_TIMED_LAUNCH(c, "k_hist2_update", 1, rr::launch_hist2_update<T>(io.in, io.in_stride, len, hin, hout, (long long)n, ncop, S, st,
                                                                                                s.hist_fused_jlo, -1));
                    } else {
                        RR_TIMED_LAUNCH(c, "k_hist2_update", 1, rr::launch_hist2_update<T>(io.in, io.in_stride, len, hin, hout, (long long)n, ncop, S, st, 0, -1));
                    }
                }
                s.hist_fused_jlo = -1;
                s.hist_cur ^= 1;
                if (io.nco) {
                    RR_LAUNCH(1, rr::launch_nco_advance((rr::NcoStream*)io.nco->nco_d.p, S, len, st));
                    nco_host_advance(*io.nco, len);
                }
                if (took_ds) ++i;  // the Downsampler stage is done
                break;
            }
            case RR_STAGE_DOWNSAMPLE:
            case RR_STAGE_UPSAMPLE: {
                const bool down = s.d.kind == RR_STAGE_DOWNSAMPLE;
                if (a.redesign) RR_TRY(resampler_redesign<T>(c, s, cur.sh.rate));
                if (synth && i == ns - 2) {
                    // Upsampler -> FreqShifter -> sum in k_synth: the Upsampler's state (carried sums, the pending part
                    // behind the last whole chunk) and the NCO advance exactly as in a per-stream push.  The staging
                    // buffers hold only the pending parts, less than one output chunk per stream.
                    const long long emit = (long long)a.out.len();
                    RR_TRY(obuf_reserve<T>(c, s, std::max<size_t>(a.pending_before, a.pending_before + a.n_new - (size_t)emit), a.pending_before));
                    Stage& fs = c->st[i + 1];
                    StageAct fa;
                    RR_TRY(advance_stage(fs.d, fs.h, a.out, &fa));
                    RR_TRY(nco_refresh<T>(c, fs, a.out.rate, fa.nco_recalc));
                    rr::SynthArgs sa{};
                    sa.in = cur.p;
                    sa.in_stride = cur.stride;
                    sa.len = len;
                    sa.acc_in = s.tail[s.tail_cur].p;
                    sa.acc_out = s.tail[s.tail_cur ^ 1].p;
                    sa.ir = s.ir.p;
                    sa.L = s.h.r_L;
                    sa.Q = (int)s.h.Q;
                    sa.j0 = a.j0;
                    sa.m0 = a.m0;
                    sa.n_new = (long long)a.n_new;
                    sa.pend = s.obuf[s.obuf_cur].p;
                    sa.pending = (long long)a.pending_before;
                    sa.rem = s.obuf[s.obuf_cur ^ 1].p;
                    sa.obuf_stride = (long long)s.obuf_cap;
                    sa.split = emit - (long long)a.pending_before;
                    sa.nco = (const rr::NcoStream*)fs.nco_d.p;
                    sa.out = dev_out;
                    sa.emit = emit;
                    RR_TIMED_LAUNCH(c, "k_synth", 1, rr::launch_synth<T>(sa, S, c->ctx->sm_count, st));
                    RR_LAUNCH(1, rr::launch_nco_advance((rr::NcoStream*)fs.nco_d.p, S, emit, st));
                    nco_host_advance(fs, emit);
                    s.tail_cur ^= 1;
                    s.obuf_cur ^= 1;  // the remainder now lives in the other staging buffer (emit > 0)
                    cur.p = dev_out;
                    cur.stride = 0;
                    cur.sh = fa.out;
                    plan += "synth[upsample+nco+sum]";
                    ++i;  // the FreqShifter stage is done
                    break;
                }
                RR_TRY(obuf_reserve<T>(c, s, a.pending_before + a.n_new, a.pending_before));
                void* o = (char*)s.obuf[s.obuf_cur].p + a.pending_before * 2 * sizeof(T);
                rr::RateState rs;
                rs.P = s.h.P;
                rs.Q = s.h.Q;
                rs.j0 = a.j0;
                rs.m0 = a.m0;
                if (s.h.r_indexed) {
                    if (down) RR_TRY(downsample_indexed<T>(c, s, a, cur.p, cur.stride, len, o, (long long)s.obuf_cap));
                    else RR_TRY(upsample_indexed<T>(c, s, a, cur.p, cur.stride, len, o, (long long)s.obuf_cap));
                    plan += down ? "downsample(indexed)" : "upsample(indexed)";
                    RR_TRY(resampler_emit<T>(c, s, a, last, dev_out, (long long)out_stride, &cur));
                    break;
                }
                if (down) {
                    RR_TIMED_LAUNCH(c, "k_downsample", 2, rr::launch_downsample<T>(cur.p, cur.stride, len, s.tail[s.tail_cur].p, s.tail[s.tail_cur ^ 1].p,
                                                          (const T*)s.ir.p, s.h.r_L, rs, (long long)a.n_new, o, (long long)s.obuf_cap, S, st));
                    plan += "downsample";
                } else {
                    // last stage: whole output chunks go straight to the caller's buffer, the part behind them to the other
                    // staging buffer (no copy of the new samples afterwards)
                    const long long emit = (long long)a.out.len();
                    bool direct = false;
                    if (last && emit > 0 && emit >= (long long)a.pending_before && rr::upsample_tiled_supported<T>(rs, s.h.r_L)) {
                        void* d1 = (char*)dev_out + a.pending_before * 2 * sizeof(T);
                        RR_TIMED_LAUNCH(c, "k_upsample", 1, rr::launch_upsample<T>(cur.p, cur.stride, len, s.tail[s.tail_cur].p, s.tail[s.tail_cur ^ 1].p,
                                                            (const T*)s.ir.p, s.h.r_L, rs, (long long)a.n_new, d1, (long long)out_stride, S, st,
                                                            s.obuf[s.obuf_cur ^ 1].p, (long long)s.obuf_cap, emit - (long long)a.pending_before));
                        direct = true;
                    } else {
                        RR_TIMED_LAUNCH(c, "k_upsample", 1, rr::launch_upsample<T>(cur.p, cur.stride, len, s.tail[s.tail_cur].p, s.tail[s.tail_cur ^ 1].p,
                                                            (const T*)s.ir.p, s.h.r_L, rs, (long long)a.n_new, o, (long long)s.obuf_cap, S, st));
                    }
                    plan += "upsample";
                    s.tail_cur ^= 1;
                    RR_TRY(resampler_emit<T>(c, s, a, last, dev_out, (long long)out_stride, &cur, direct));
                    break;
                }
                s.tail_cur ^= 1;
                RR_TRY(resampler_emit<T>(c, s, a, last, dev_out, (long long)out_stride, &cur));
                break;
            }
            default:
                return fail(RR_ERR_INVALID, "unknown stage kind");
        }
    }
    // a chain whose last active stage did not write into the caller's buffer
    // (inactive tail stages, or an empty chain): copy the samples through
    if (cur.sh.len() > 0 && cur.p != dev_out) {
        RR_LAUNCH(1, rr::launch_copy2d<T>(cur.p, cur.stride, dev_out, (long long)out_stride, (long long)cur.sh.len(), S, st));
    }
    if (summed && !synth && cur.sh.len() > 0) {
        RR_TIMED_LAUNCH(c, "k_stream_sum", 1, rr::launch_stream_sum<T>(dev_out, (long long)out_stride, (long long)cur.sh.len(), S, row_out, st));
        plan += "|sum";
    }
    if (out_count) *out_count = cur.sh.len();
    if (out_rate) *out_rate = cur.sh.rate;
    c->plan = plan;
    return RR_OK;
}

// every block back to its state after construction; parameters (shifts, responses, deviations, gains) are kept
void chain_restart(rr_chain* c) {
    for (auto& s : c->st) {
        s.h = StageHost{};
        s.taps_valid = false;
        s.poly_valid = s.poly_tried = s.poly2_valid = s.front_valid = s.frontq_valid = false;
        s.ztail_stale = false;
        s.ucache_valid = false;
        s.hist_fused_jlo = -1;
        s.fwin_n = 0;
        for (auto& h : s.nco_h) h = NcoHost{};
        if (s.d.kind == RR_STAGE_FREQSHIFT) {
            std::fill(s.shift_dirty.begin(), s.shift_dirty.end(), (uint8_t)1);
            s.any_shift_dirty = true;
        }
        // FmMod's phase accumulator restarts at zero like a new block's
        if (s.fm_phase.p) cudaMemsetAsync(s.fm_phase.p, 0, s.fm_phase.bytes, c->stream);
        if (s.fm_last.p) cudaMemsetAsync(s.fm_last.p, 0, s.fm_last.bytes, c->stream);
    }
}

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

const char* rr_last_error(void) { return g_err.c_str(); }

int rr_version(int* major, int* minor) {
    if (major) *major = RR_VERSION_MAJOR;
    if (minor) *minor = RR_VERSION_MINOR;
    return RR_OK;
}

uint64_t rr_kernel_launch_count(void) { return g_launches.load(); }

int rr_ctx_create(int device, rr_ctx** out) {
    if (!out) return fail(RR_ERR_INVALID, "rr_ctx_create: out is null");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(RR_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(RR_ERR_INVALID, "rr_ctx_create: device index out of range");
    RR_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0)  // sm_100a SASS is architecture specific and ships without PTX
        return fail(RR_ERR_UNSUPPORTED, "this library holds sm_100a code only; the device's compute capability is not 10.0");
    rr_ctx* c = new rr_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    *out = c;
    return RR_OK;
}
int rr_ctx_destroy(rr_ctx* ctx) {
    delete ctx;
    return RR_OK;
}
int rr_ctx_device(const rr_ctx* ctx) { return ctx ? ctx->device : -1; }

int rr_pinned_alloc(rr_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return fail(RR_ERR_INVALID, "rr_pinned_alloc: null argument");
    RR_CUDA(cudaSetDevice(ctx->device));
    RR_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return RR_OK;
}
int rr_pinned_free(rr_ctx* ctx, void* p) {
    if (!ctx) return fail(RR_ERR_INVALID, "rr_pinned_free: null context");
    if (p) RR_CUDA(cudaFreeHost(p));
    return RR_OK;
}
int rr_host_register(rr_ctx* ctx, void* p, size_t bytes) {
    if (!ctx || !p) return fail(RR_ERR_INVALID, "rr_host_register: null argument");
    RR_CUDA(cudaSetDevice(ctx->device));
    RR_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return RR_OK;
}
int rr_host_unregister(rr_ctx* ctx, void* p) {
    if (!ctx || !p) return fail(RR_ERR_INVALID, "rr_host_unregister: null argument");
    RR_CUDA(cudaHostUnregister(p));
    return RR_OK;
}
// ---- pinned chunk pool (bufferpool.rs:187-222) -----------------------------------
int rr_pool_create(rr_ctx* ctx, rr_pool** out) {
    if (!ctx || !out) return fail(RR_ERR_INVALID, "rr_pool_create: null argument");
    rr_pool* p = new rr_pool();
    p->ctx = ctx;
    *out = p;
    return RR_OK;
}
int rr_pool_get(rr_pool* pool, size_t min_bytes, void** out, size_t* capacity) {
    if (!pool || !out) return fail(RR_ERR_INVALID, "rr_pool_get: null argument");
    *out = nullptr;
    RR_CUDA(cudaSetDevice(pool->ctx->device));
    const size_t need = min_bytes ? min_bytes : 1;
    void* small = nullptr;
    {
        // ChunkBufPool::get_with_capacity takes the oldest recycled buffer (bufferpool.rs:213-216); a Vec that is too
        // small grows when it is filled -- pinned memory cannot, so a too-small buffer is replaced here
        std::lock_guard<std::mutex> lk(pool->mu);
        if (!pool->idle.empty()) {
            rr_pool::Buf b = pool->idle.front();
            pool->idle.pop_front();
            if (b.cap >= need) {
                pool->live[b.p] = b.cap;
                ++pool->n_reuse;
                *out = b.p;
                if (capacity) *capacity = b.cap;
                return RR_OK;
            }
            small = b.p;
        }
    }
    if (small) cudaFreeHost(small);
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, need, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? RR_ERR_NOMEM : RR_ERR_CUDA, std::string("rr_pool_get: cudaHostAlloc: ") + cudaGetErrorString(e));
    }
    std::lock_guard<std::mutex> lk(pool->mu);
    pool->live[p] = need;
    ++pool->n_alloc;
    *out = p;
    if (capacity) *capacity = need;
    return RR_OK;
}
int rr_pool_put(rr_pool* pool, void* p) {
    if (!pool) return fail(RR_ERR_INVALID, "rr_pool_put: null pool");
    if (!p) return RR_OK;
    std::lock_guard<std::mutex> lk(pool->mu);
    auto it = pool->live.find(p);
    if (it == pool->live.end()) return fail(RR_ERR_INVALID, "rr_pool_put: the buffer is not on loan from this pool");
    pool->idle.push_back(rr_pool::Buf{p, it->second});
    pool->live.erase(it);
    return RR_OK;
}
int rr_pool_stats(rr_pool* pool, uint64_t* allocated, uint64_t* reused, uint64_t* idle_buffers, uint64_t* live_buffers) {
    if (!pool) return fail(RR_ERR_INVALID, "rr_pool_stats: null pool");
    std::lock_guard<std::mutex> lk(pool->mu);
    if (allocated) *allocated = pool->n_alloc;
    if (reused) *reused = pool->n_reuse;
    if (idle_buffers) *idle_buffers = pool->idle.size();
    if (live_buffers) *live_buffers = pool->live.size();
    return RR_OK;
}
int rr_pool_trim(rr_pool* pool) {
    if (!pool) return fail(RR_ERR_INVALID, "rr_pool_trim: null pool");
    std::deque<rr_pool::Buf> drop;
    {
        std::lock_guard<std::mutex> lk(pool->mu);
        drop.swap(pool->idle);
    }
    for (auto& b : drop) cudaFreeHost(b.p);
    return RR_OK;
}
int rr_pool_destroy(rr_pool* pool) {
    if (!pool) return RR_OK;
    rr_pool_trim(pool);
    // buffers still on loan die with the pool, like Chunks that outlive their ChunkBufPool lose their recycler
    // (bufferpool.rs:85-88: a closed channel makes the send fail and the Vec is dropped)
    for (auto& kv : pool->live) cudaFreeHost(kv.first);
    delete pool;
    return RR_OK;
}
int rr_device_alloc(rr_ctx* ctx, size_t bytes, void** out) {
    if (!ctx || !out) return fail(RR_ERR_INVALID, "rr_device_alloc: null argument");
    RR_CUDA(cudaSetDevice(ctx->device));
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 16);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return fail(RR_ERR_NOMEM, "rr_device_alloc: out of device memory");
    }
    RR_CUDA(e);
    return RR_OK;
}
int rr_device_free(rr_ctx* ctx, void* p) {
    if (!ctx) return fail(RR_ERR_INVALID, "rr_device_free: null context");
    RR_CUDA(cudaSetDevice(ctx->device));
    if (p) RR_CUDA(cudaFree(p));
    return RR_OK;
}
// ---- device buffers shared between processes (one process per GPU): the gather of the channelizer outputs -------
int rr_ipc_export(rr_ctx* ctx, void* dev_ptr, void* handle_out_64_bytes) {
    if (!ctx || !dev_ptr || !handle_out_64_bytes) return fail(RR_ERR_INVALID, "rr_ipc_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the header promises a 64-byte handle");
    RR_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    RR_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
    std::memcpy(handle_out_64_bytes, &h, sizeof h);
    return RR_OK;
}
int rr_ipc_open(rr_ctx* ctx, const void* handle_64_bytes, void** dev_ptr) {
    if (!ctx || !handle_64_bytes || !dev_ptr) return fail(RR_ERR_INVALID, "rr_ipc_open: null argument");
    *dev_ptr = nullptr;
    RR_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle_64_bytes, sizeof h);
    RR_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return RR_OK;
}
int rr_ipc_close(rr_ctx* ctx, void* dev_ptr) {
    if (!ctx) return fail(RR_ERR_INVALID, "rr_ipc_close: null context");
    RR_CUDA(cudaSetDevice(ctx->device));
    if (dev_ptr) RR_CUDA(cudaIpcCloseMemHandle(dev_ptr));
    return RR_OK;
}
int rr_memcpy_h2d(rr_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes) {
    if (!ctx) return fail(RR_ERR_INVALID, "rr_memcpy_h2d: null context");
    RR_CUDA(cudaSetDevice(ctx->device));
    RR_CUDA(cudaDeviceSynchronize());  // chains run on non-blocking streams: nothing may still be reading dst_dev
    RR_CUDA(cudaMemcpy(dst_dev, src_host, bytes, cudaMemcpyHostToDevice));
    return RR_OK;
}
int rr_memcpy_d2h(rr_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes) {
    if (!ctx) return fail(RR_ERR_INVALID, "rr_memcpy_d2h: null context");
    RR_CUDA(cudaSetDevice(ctx->device));
    RR_CUDA(cudaDeviceSynchronize());  // src_dev may still be written by a chain's (non-blocking) stream
    RR_CUDA(cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost));
    return RR_OK;
}

// ---- metering (src/metering.rs:21-30) ---------------------------------------------
int rr_metering_level(rr_ctx* ctx, int32_t dtype, const void* dev_in, size_t in_stride, size_t chunk_len, size_t n_chunks, int n_streams,
                      double* host_out) {
    if (!ctx || !host_out || (!dev_in && n_chunks)) return fail(RR_ERR_INVALID, "rr_metering_level: null argument");
    if (dtype != RR_C32 && dtype != RR_C64) return fail(RR_ERR_INVALID, "rr_metering_level: bad dtype");
    if (n_streams < 1 || chunk_len == 0) return fail(RR_ERR_INVALID, "rr_metering_level: empty chunk (the reference divides by zero)");
    if (n_streams > 65535) return fail(RR_ERR_INVALID, "rr_metering_level: at most 65535 streams per call");
    if (n_chunks == 0) return RR_OK;
    RR_CUDA(cudaSetDevice(ctx->device));
    (void)cudaGetLastError();  // a stale error of an unrelated earlier call is not ours
    RR_CUDA(cudaDeviceSynchronize());  // dev_in may still be written by a chain's (non-blocking) stream
    DevBuf out;
    RR_TRY(out.ensure(sizeof(double) * n_chunks * (size_t)n_streams));
    cudaError_t e = dtype == RR_C32 ? rr::launch_level<float>(dev_in, (long long)in_stride, (long long)chunk_len, (long long)n_chunks, n_streams,
                                                              (double*)out.p, nullptr)
                                    : rr::launch_level<double>(dev_in, (long long)in_stride, (long long)chunk_len, (long long)n_chunks, n_streams,
                                                               (double*)out.p, nullptr);
    if (e == cudaSuccess) {
        g_launches.fetch_add(1);
        e = cudaMemcpy(host_out, out.p, sizeof(double) * n_chunks * (size_t)n_streams, cudaMemcpyDeviceToHost);
    }
    out.release();
    if (e != cudaSuccess) return fail_cuda(e, "rr_metering_level");
    return RR_OK;
}

int rr_metering_bandwidth(rr_ctx* ctx, int32_t dtype, const void* dev_bins, size_t in_stride, size_t chunk_len, size_t n_chunks,
                          int n_streams, double double_percentile, double sample_rate, double* host_out) {
    if (!ctx || !host_out || (!dev_bins && n_chunks)) return fail(RR_ERR_INVALID, "rr_metering_bandwidth: null argument");
    if (dtype != RR_C32 && dtype != RR_C64) return fail(RR_ERR_INVALID, "rr_metering_bandwidth: bad dtype");
    if (n_streams < 1 || n_streams > 65535 || chunk_len == 0) return fail(RR_ERR_INVALID, "rr_metering_bandwidth: empty chunk or bad stream count");
    if (n_chunks == 0) return RR_OK;
    RR_CUDA(cudaSetDevice(ctx->device));
    (void)cudaGetLastError();  // a stale error of an unrelated earlier call is not ours
    RR_CUDA(cudaDeviceSynchronize());  // dev_bins may still be written by a chain's (non-blocking) stream
    DevBuf out;
    RR_TRY(out.ensure(sizeof(double) * n_chunks * (size_t)n_streams));
    cudaError_t e = dtype == RR_C32 ? rr::launch_bandwidth<float>(dev_bins, (long long)in_stride, (long long)chunk_len, (long long)n_chunks, n_streams,
                                                                  double_percentile, sample_rate, (double*)out.p, nullptr)
                                    : rr::launch_bandwidth<double>(dev_bins, (long long)in_stride, (long long)chunk_len, (long long)n_chunks, n_streams,
                                                                   double_percentile, sample_rate, (double*)out.p, nullptr);
    if (e == cudaSuccess) {
        g_launches.fetch_add(1);
        e = cudaMemcpy(host_out, out.p, sizeof(double) * n_chunks * (size_t)n_streams, cudaMemcpyDeviceToHost);
    }
    out.release();
    if (e != cudaSuccess) return fail_cuda(e, "rr_metering_bandwidth");
    return RR_OK;
}

int rr_metering_rescale_energy(rr_ctx* ctx, int32_t dtype, const void* dev_bins, size_t in_stride, size_t chunk_len, size_t n_chunks,
                               int n_streams, size_t resolution, void* host_out) {
    if (!ctx || !host_out || (!dev_bins && n_chunks)) return fail(RR_ERR_INVALID, "rr_metering_rescale_energy: null argument");
    if (dtype != RR_C32 && dtype != RR_C64) return fail(RR_ERR_INVALID, "rr_metering_rescale_energy: bad dtype");
    if (chunk_len == 0) return fail(RR_ERR_INVALID, "rr_metering_rescale_energy: empty input (metering.rs:98 asserts n > 0)");
    if (n_streams < 1 || n_streams > 65535 || n_chunks > 65535) return fail(RR_ERR_INVALID, "rr_metering_rescale_energy: at most 65535 streams and chunks per call");
    if (n_chunks == 0 || resolution == 0) return RR_OK;
    RR_CUDA(cudaSetDevice(ctx->device));
    (void)cudaGetLastError();  // a stale error of an unrelated earlier call is not ours
    RR_CUDA(cudaDeviceSynchronize());  // dev_bins may still be written by a chain's (non-blocking) stream
    const size_t fsz = dtype == RR_C32 ? sizeof(float) : sizeof(double);
    const size_t bytes = fsz * n_chunks * (size_t)n_streams * resolution;
    DevBuf out;
    RR_TRY(out.ensure(bytes));
    cudaError_t e = dtype == RR_C32 ? rr::launch_rescale_energy<float>(dev_bins, (long long)in_stride, (long long)chunk_len, (long long)n_chunks,
                                                                       n_streams, (long long)resolution, out.p, nullptr)
                                    : rr::launch_rescale_energy<double>(dev_bins, (long long)in_stride, (long long)chunk_len, (long long)n_chunks,
                                                                        n_streams, (long long)resolution, out.p, nullptr);
    if (e == cudaSuccess) {
        g_launches.fetch_add(1);
        e = cudaMemcpy(host_out, out.p, bytes, cudaMemcpyDeviceToHost);
    }
    out.release();
    if (e != cudaSuccess) return fail_cuda(e, "rr_metering_rescale_energy");
    return RR_OK;
}

// ---- design math ------------------------------------------------------------
double rr_bessel_i0(double x) { return rr::bessel_i0(x); }
double rr_sinc(double x) { return rr::sinc(x); }
double rr_kaiser_rel_with_beta(double beta, double x) { return rr::kaiser_rel_with_beta(beta, x); }
double rr_kaiser_null_at_bin_to_beta(double n) { return rr::kaiser_null_at_bin_to_beta(n); }
void rr_deemphasis_factor(double tau, double frequency, double* out_re, double* out_im) {
    const std::complex<double> v = rr::deemphasis_factor(tau, frequency);
    if (out_re) *out_re = v.real();
    if (out_im) *out_im = v.imag();
}
int rr_freq_to_ratio(double sample_rate, double precision, double frequency, int64_t* numer, int64_t* denom) {
    int64_t n = 0, d = 1;
    if (!rr::freq_to_ratio(sample_rate, precision, frequency, &n, &d))
        return fail(RR_ERR_INVALID, "denominator == 0 (Ratio::new panics in the reference)");
    if (numer) *numer = n;
    if (denom) *denom = d;
    return RR_OK;
}
int rr_design_filter_response(rr_freq_resp_fn f, void* f_user, int32_t window_kind, double window_beta, rr_window_fn w, void* w_user,
                              double sample_rate, size_t n, int32_t dtype, double* out_2n_complex) {
    if (!f || !out_2n_complex) return fail(RR_ERR_INVALID, "rr_design_filter_response: null argument");
    rr::FreqResp fr = [f, f_user](int64_t bin, double freq) {
        double re = 0.0, im = 0.0;
        f(f_user, bin, freq, &re, &im);
        return std::complex<double>(re, im);
    };
    std::vector<std::complex<double>> H;
    if (!rr::design_filter_response(fr, make_window(window_kind, window_beta, w, w_user), sample_rate, n, dtype == RR_C32, &H))
        return fail(RR_ERR_INVALID, "rr_design_filter_response: n must be >= 1");
    for (size_t i = 0; i < H.size(); ++i) {
        out_2n_complex[2 * i] = H[i].real();
        out_2n_complex[2 * i + 1] = H[i].imag();
    }
    return RR_OK;
}
static int design_taps(bool down, double input_rate, double output_rate, double bandwidth, double quality, size_t* ir_len, double* ir) {
    if (!ir_len) return fail(RR_ERR_INVALID, "ir_len is null");
    if (!(output_rate >= 0.0) || !(bandwidth >= 0.0) || !(input_rate >= 0.0)) return fail(RR_ERR_INVALID, "rates must be positive");
    if (down && !(bandwidth < output_rate)) return fail(RR_ERR_INVALID, "bandwidth must be smaller than output sample rate");
    if (down && !(input_rate >= output_rate)) return fail(RR_ERR_INVALID, "input sample rate must be >= output sample rate");
    if (!down && !(input_rate <= output_rate)) return fail(RR_ERR_INVALID, "input sample rate must be <= output sample rate");
    if (!down && !(bandwidth < input_rate)) return fail(RR_ERR_INVALID, "bandwidth must be smaller than input sample rate");
    const double margin = down ? (output_rate - bandwidth) / 2.0 : (input_rate - bandwidth) / 2.0;
    const double lf = std::ceil((down ? input_rate : output_rate) / margin * quality);
    if (!(lf > 0.0) || lf > 1.0e8) return fail(RR_ERR_INVALID, "impulse response length out of range");
    const size_t L = (size_t)lf;
    const size_t cap = *ir_len;
    *ir_len = L;
    if (!ir) return RR_OK;
    if (cap < L) return fail(RR_ERR_CAPACITY, "ir buffer too small");
    std::vector<double> taps;
    const double ratio = down ? output_rate / input_rate : input_rate / output_rate;
    const double null_bin = (double)L * margin / (down ? input_rate : output_rate);
    rr::design_resampler_taps(L, ratio, null_bin, &taps);
    std::memcpy(ir, taps.data(), L * sizeof(double));
    return RR_OK;
}
int rr_design_downsampler_taps(double input_rate, double output_rate, double bandwidth, double quality, size_t* ir_len, double* ir) {
    return design_taps(true, input_rate, output_rate, bandwidth, quality, ir_len, ir);
}
int rr_design_upsampler_taps(double input_rate, double output_rate, double bandwidth, double quality, size_t* ir_len, double* ir) {
    return design_taps(false, input_rate, output_rate, bandwidth, quality, ir_len, ir);
}

// Rank of the fused Filter -> Downsampler filter for integer decimation (rr_design.h: design_rank_tables),
// the part it discards, and how far sum_c a_c b_c^T is from the full polyphase tables (relative L2 over
// all P*K table entries) -- the last one is the check that the factorisation is exact to rounding.
int rr_design_fused_rank(rr_freq_resp_fn f, void* f_user, int32_t window_kind, double window_beta, rr_window_fn w, void* w_user,
                         double sample_rate, size_t n, double output_rate, double bandwidth, double quality, double tol, int max_rank,
                         int* rank, double* discarded, double* table_error) {
    if (!f || !rank) return fail(RR_ERR_INVALID, "rr_design_fused_rank: null argument");
    if (max_rank < 1 || max_rank > 64) return fail(RR_ERR_INVALID, "rr_design_fused_rank: max_rank out of range");
    rr::FreqResp fr = [f, f_user](int64_t bin, double freq) {
        double re = 0.0, im = 0.0;
        f(f_user, bin, freq, &re, &im);
        return std::complex<double>(re, im);
    };
    std::vector<std::complex<double>> resp, taps;
    if (!is_pow2(n)) return fail(RR_ERR_INVALID, "rr_design_fused_rank: the fused kernels run on power-of-two chunk lengths >= 2");
    if (!rr::design_filter_response(fr, make_window(window_kind, window_beta, w, w_user), sample_rate, n, true, &resp, &taps))
        return fail(RR_ERR_INVALID, "rr_design_fused_rank: filter design failed");
    if (!integer_valued(sample_rate) || !integer_valued(output_rate) || output_rate <= 0.0 || sample_rate < output_rate)
        return fail(RR_ERR_INVALID, "rr_design_fused_rank: rates must be integer valued, input >= output > 0");
    const long long g = std::gcd((long long)sample_rate, (long long)output_rate);
    const long long P = (long long)sample_rate / g, Q = (long long)output_rate / g;
    if (Q < 1 || Q > 4) return fail(RR_ERR_UNSUPPORTED, "rr_design_fused_rank: in/out = P/Q with Q <= 4 only");
    size_t L = 0;
    RR_TRY(design_taps(true, sample_rate, output_rate, bandwidth, quality, &L, nullptr));
    std::vector<double> ir(L);
    RR_TRY(design_taps(true, sample_rate, output_rate, bandwidth, quality, &L, ir.data()));
    for (auto& v : ir) v = (double)(float)v;
    const int K = 512;
    std::vector<double> a;
    std::vector<std::complex<double>> b, full;
    double disc = 0.0;
    // Q == 1: b is [max_rank][K]; Q > 1: the phases factored together, b is [Q][max_rank][K]
    const int lmax = Q == 1 ? rr::design_rank_tables(taps, ir, P, K, tol, max_rank, rank, &a, &b, &disc)
                            : rr::design_rank_tables_q(taps, ir, P, Q, K, tol, max_rank, rank, &a, &b, &disc);
    if (discarded) *discarded = disc;
    if (table_error) {
        *table_error = -1.0;
        if (*rank > 0 && lmax + 2 <= K) {
            rr::design_poly_tables(taps, ir, P, Q, K, &full);
            double num = 0.0, den = 0.0;
            for (long long q = 0; q < Q; ++q)
                for (long long p = 0; p < P; ++p)
                    for (int k = 0; k < K; ++k) {
                        std::complex<double> sum(0.0, 0.0);
                        for (int c = 0; c < *rank; ++c) sum += a[(size_t)p * max_rank + c] * b[((size_t)q * max_rank + c) * K + k];
                        const std::complex<double> want = full[(size_t)(q * P + p) * K + k];
                        num += std::norm(sum - want);
                        den += std::norm(want);
                    }
            *table_error = den > 0.0 ? std::sqrt(num / den) : 0.0;
        }
    }
    return RR_OK;
}

// ---- chain ---------------------------------------------------------------------
int rr_chain_create(rr_ctx* ctx, const rr_chain_desc* desc, rr_chain** out) {
    if (!ctx || !desc || !out) return fail(RR_ERR_INVALID, "rr_chain_create: null argument");
    *out = nullptr;
    if (desc->dtype != RR_C32 && desc->dtype != RR_C64) return fail(RR_ERR_INVALID, "rr_chain_create: bad dtype");
    if (desc->n_streams < 1) return fail(RR_ERR_INVALID, "rr_chain_create: n_streams must be >= 1");
    if (desc->n_streams > 65535) return fail(RR_ERR_INVALID, "rr_chain_create: at most 65535 streams per chain (streams map to a grid dimension)");
    if (desc->n_stages < 0 || (desc->n_stages > 0 && !desc->stages)) return fail(RR_ERR_INVALID, "rr_chain_create: bad stage list");
    for (int i = 0; i < desc->n_stages; ++i) {
        const rr_stage_desc& d = desc->stages[i];
        switch (d.kind) {
            case RR_STAGE_FREQSHIFT:
                if (!(d.precision > 0.0)) return fail(RR_ERR_INVALID, "FreqShifter: precision must be positive");
                break;
            case RR_STAGE_FILTER:
                if (!d.freq_resp) return fail(RR_ERR_INVALID, "Filter: freq_resp callback is null");
                break;
            case RR_STAGE_DOWNSAMPLE:  // resampling.rs:51-56
                if (!(d.output_rate >= 0.0)) return fail(RR_ERR_INVALID, "output sample rate must be positive");
                if (!(d.bandwidth >= 0.0)) return fail(RR_ERR_INVALID, "bandwidth must be positive");
                if (!(d.bandwidth < d.output_rate)) return fail(RR_ERR_INVALID, "bandwidth must be smaller than output sample rate");
                if (!(d.quality >= 1.0)) return fail(RR_ERR_INVALID, "quality must be >= 1.0");
                break;
            case RR_STAGE_UPSAMPLE:  // resampling.rs:186-188
                if (!(d.output_rate >= 0.0)) return fail(RR_ERR_INVALID, "output sample rate must be positive");
                if (!(d.bandwidth >= 0.0)) return fail(RR_ERR_INVALID, "bandwidth must be positive");
                if (!(d.quality >= 1.0)) return fail(RR_ERR_INVALID, "quality must be >= 1.0");
                break;
            case RR_STAGE_FMDEMOD:
            case RR_STAGE_FMMOD:
            case RR_STAGE_GAIN:
            case RR_STAGE_FOURIER:
                break;
            case RR_STAGE_RECHUNK:  // chunks.rs:58
                if (d.output_chunk_len == 0) return fail(RR_ERR_INVALID, "chunk length must be positive");
                break;
            case RR_STAGE_OVERLAP:  // chunks.rs:195
                if (d.chunk_count <= 0) return fail(RR_ERR_INVALID, "chunk count must be positive");
                break;
            default:
                return fail(RR_ERR_INVALID, "rr_chain_create: unknown stage kind");
        }
    }
    RR_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<rr_chain> c(new rr_chain());
    c->ctx = ctx;
    c->dtype = desc->dtype;
    c->esz = desc->dtype == RR_C32 ? 8 : 16;
    c->S = desc->n_streams;
    c->st.resize((size_t)desc->n_stages);
    for (int i = 0; i < desc->n_stages; ++i) {
        Stage& s = c->st[(size_t)i];
        s.d = desc->stages[i];
        if (s.d.kind == RR_STAGE_FREQSHIFT) {
            s.shift.assign((size_t)c->S, s.d.shift);
            s.shift_dirty.assign((size_t)c->S, 1);
            s.any_shift_dirty = true;
        }
    }
    if (const char* e = std::getenv("RR_DISABLE_POLY")) c->allow_poly = !(e[0] == '1');
    if (const char* e = std::getenv("RR_DISABLE_POLY2")) c->allow_poly2 = !(e[0] == '1');
    if (const char* e = std::getenv("RR_DISABLE_FRONT")) c->allow_front = !(e[0] == '1');
    if (const char* e = std::getenv("RR_DISABLE_FUSED")) c->allow_fused = !(e[0] == '1');
    c->fused_min_streams = 2 * ctx->sm_count;
    if (const char* e = std::getenv("RR_FUSED_MIN_STREAMS")) c->fused_min_streams = std::max(1, std::atoi(e));
    if (const char* e = std::getenv("RR_FUSED_MIN_ROWS")) c->fused_min_rows = std::max(1, std::atoi(e));
    if (const char* e = std::getenv("RR_DISABLE_UCACHE")) c->allow_ucache = !(e[0] == '1');
    if (const char* e = std::getenv("RR_DISABLE_SAB")) c->allow_sab = !(e[0] == '1');
    if (const char* e = std::getenv("RR_BIG_OS_SCRATCH_MB")) c->big_os_scratch_bytes = (size_t)std::max(1, std::atoi(e)) << 20;
    RR_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    *out = c.release();
    return RR_OK;
}

int rr_chain_destroy(rr_chain* c) {
    if (!c) return RR_OK;
    cudaSetDevice(c->ctx->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (auto& s : c->st) {
        DevBuf* bufs[] = {&s.nco_d, &s.hperm, &s.tw, &s.hist2[0], &s.hist2[1], &s.ztmp, &s.gtab, &s.twK, &s.big_h, &s.big_twA, &s.big_twB, &s.big_twC, &s.big_scratch,
                          &s.ir, &s.tail[0], &s.tail[1], &s.obuf[0], &s.obuf[1], &s.fm_prev, &s.fm_last, &s.out,
                          &s.gtab2, &s.twK2, &s.acoef, &s.gtab3, &s.acoef_q, &s.gtab_q, &s.ubuf[0], &s.ubuf[1], &s.fwin, &s.ftw, &s.fm_phase, &s.ukeep[0], &s.ukeep[1],
                          &s.stg_in, &s.stg_out, &s.zero_chunk, &s.idx_a, &s.idx_b};
        for (DevBuf* b : bufs) b->release();
        if (s.fused_slot >= 0) fused_slot_release(c->ctx->device, &s);
    }
    c->sum_rows.release();
    if (c->d2h_stream) cudaStreamSynchronize(c->d2h_stream);
    if (c->h2d_stream) cudaStreamSynchronize(c->h2d_stream);
    for (int k = 0; k < 2; ++k) {
        c->stage_in[k].release();
        c->stage_out[k].release();
        if (c->ev_h2d[k]) cudaEventDestroy(c->ev_h2d[k]);
        if (c->ev_comp[k]) cudaEventDestroy(c->ev_comp[k]);
        if (c->ev_d2h[k]) cudaEventDestroy(c->ev_d2h[k]);
    }
    for (cudaEvent_t e : c->evs) cudaEventDestroy(e);
    if (c->ev_copy) cudaEventDestroy(c->ev_copy);
    if (c->h2d_stream) cudaStreamDestroy(c->h2d_stream);
    if (c->d2h_stream) cudaStreamDestroy(c->d2h_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return RR_OK;
}

static int stage_of(rr_chain* c, int stage, int kind, Stage** out) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    if (stage < 0 || stage >= (int)c->st.size()) return fail(RR_ERR_INVALID, "stage index out of range");
    if (c->st[(size_t)stage].d.kind != kind) return fail(RR_ERR_INVALID, "stage is of a different kind");
    *out = &c->st[(size_t)stage];
    return RR_OK;
}

int rr_chain_set_shift(rr_chain* c, int stage, int stream, double shift_hz) {
    Stage* s = nullptr;
    RR_TRY(stage_of(c, stage, RR_STAGE_FREQSHIFT, &s));
    if (stream >= c->S) return fail(RR_ERR_INVALID, "stream index out of range");
    if (stream < 0) {
        for (int i = 0; i < c->S; ++i) {
            s->shift[(size_t)i] = shift_hz;
            s->shift_dirty[(size_t)i] = 1;
        }
    } else {
        s->shift[(size_t)stream] = shift_hz;
        s->shift_dirty[(size_t)stream] = 1;
    }
    s->any_shift_dirty = true;
    return RR_OK;
}
int rr_chain_set_shifts(rr_chain* c, int stage, const double* shifts_hz, int n) {
    Stage* s = nullptr;
    RR_TRY(stage_of(c, stage, RR_STAGE_FREQSHIFT, &s));
    if (!shifts_hz || n != c->S) return fail(RR_ERR_INVALID, "rr_chain_set_shifts: need one shift per stream");
    for (int i = 0; i < n; ++i) {
        s->shift[(size_t)i] = shifts_hz[i];
        s->shift_dirty[(size_t)i] = 1;
    }
    s->any_shift_dirty = true;
    return RR_OK;
}
int rr_chain_get_shift(rr_chain* c, int stage, int stream, double* shift_hz) {
    Stage* s = nullptr;
    RR_TRY(stage_of(c, stage, RR_STAGE_FREQSHIFT, &s));
    if (stream < 0 || stream >= c->S || !shift_hz) return fail(RR_ERR_INVALID, "bad stream index");
    *shift_hz = s->shift[(size_t)stream];
    return RR_OK;
}

int rr_chain_update_filter(rr_chain* c, int stage, rr_freq_resp_fn f, void* f_user, int32_t window_kind, double window_beta,
                           rr_window_fn w, void* w_user, int keep_window) {
    Stage* s = nullptr;
    RR_TRY(stage_of(c, stage, RR_STAGE_FILTER, &s));
    if (!f) return fail(RR_ERR_INVALID, "rr_chain_update_filter: freq_resp is null");
    s->d.freq_resp = f;
    s->d.freq_resp_user = f_user;
    if (!keep_window) {
        s->d.window_kind = window_kind;
        s->d.window_beta = window_beta;
        s->d.window_fn = w;
        s->d.window_user = w_user;
    }
    s->h.f_dirty = true;
    return RR_OK;
}
int rr_chain_set_deviation(rr_chain* c, int stage, double deviation) {
    Stage* s = nullptr;
    if (c && stage >= 0 && stage < (int)c->st.size() && c->st[(size_t)stage].d.kind == RR_STAGE_FMMOD) RR_TRY(stage_of(c, stage, RR_STAGE_FMMOD, &s));
    else RR_TRY(stage_of(c, stage, RR_STAGE_FMDEMOD, &s));
    s->d.deviation = deviation;
    return RR_OK;
}
int rr_chain_set_output_chunk_len(rr_chain* c, int stage, size_t output_chunk_len) {
    Stage* s = nullptr;
    RR_TRY(stage_of(c, stage, RR_STAGE_RECHUNK, &s));
    if (output_chunk_len == 0) return fail(RR_ERR_INVALID, "chunk length must be positive");  // chunks.rs:172
    s->d.output_chunk_len = output_chunk_len;
    return RR_OK;
}
int rr_chain_set_gain(rr_chain* c, int stage, double gain) {
    Stage* s = nullptr;
    RR_TRY(stage_of(c, stage, RR_STAGE_GAIN, &s));
    s->d.gain = gain;
    return RR_OK;
}

int rr_chain_event(rr_chain* c, int is_interrupt) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    // plain events pass every block untouched until a Rechunker / Overlapper turns them into an interrupt
    bool intr = is_interrupt != 0;
    for (auto& s : c->st) {
        c->samples_lost += (uint64_t)stage_event(s.d, s.h, &intr);
        if (intr) s.ucache_valid = false;  // the Filter in front starts a new segment
    }
    return RR_OK;
}
uint64_t rr_chain_samples_lost_count(rr_chain* c) { return c ? c->samples_lost : 0; }

size_t rr_chain_max_output(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks) {
    if (!c) return 0;
    Shape sh;
    sh.chunk_len = chunk_len;
    sh.n_chunks = n_chunks;
    sh.rate = sample_rate;
    Shape out;
    if (dry_shape(c, sh, &out) != RR_OK) return 0;
    return out.len();
}

}  // extern "C"

namespace {

// rr_chain_push_device / rr_chain_push_shared_device (shared: one input row for every stream, in_stride ignored) /
// rr_chain_push_summed_device (summed: one output row, the sum over streams; out_stride ignored)
int push_device(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in, size_t in_stride, bool shared,
                bool summed, void* dev_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    if (out_count) *out_count = 0;
    if (n_chunks == 0 || chunk_len == 0) return RR_OK;
    if (!dev_in)
        return fail(RR_ERR_INVALID, shared ? "rr_chain_push_shared_device: dev_in is null"
                                           : (summed ? "rr_chain_push_summed_device: dev_in is null" : "rr_chain_push_device: dev_in is null"));
    if (chunk_len > (size_t)1 << 30 || n_chunks > (size_t)1 << 30) return fail(RR_ERR_INVALID, "push too large");
    RR_CUDA(cudaSetDevice(c->ctx->device));
    (void)cudaGetLastError();  // a stale error of an unrelated earlier call (another library in the process) is not ours
    c->push_mutated = false;
    int r;
    if (c->dtype == RR_C32)
        r = run_push<float>(c, sample_rate, chunk_len, n_chunks, dev_in, in_stride, shared, summed, dev_out, out_capacity, out_stride,
                            out_count, out_sample_rate);
    else
        r = run_push<double>(c, sample_rate, chunk_len, n_chunks, dev_in, in_stride, shared, summed, dev_out, out_capacity, out_stride,
                             out_count, out_sample_rate);
    if (r != RR_OK && c->push_mutated) {
        // A failure behind the dry run (allocation, CUDA error) left some stages advanced and others not.  The stream
        // cannot be continued consistently: every block restarts as after rr_chain_create (parameters kept; Filters
        // redesign and prime again, resamplers restart their ring, the NCO re-derives its table at the next push).
        const std::string msg = g_err;
        chain_restart(c);
        g_err = msg + " (the chain's streaming state was reset)";
        if (out_count) *out_count = 0;
    }
    c->push_mutated = false;
    return r;
}

// rr_chain_push / rr_chain_push_shared (shared: one input row of len samples is staged and read by every stream) /
// rr_chain_push_summed (summed: one output row of max_out samples is staged and copied back)
int push_host(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* host_in, size_t in_stride, bool shared,
              bool summed, void* host_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    if (out_count) *out_count = 0;
    if (n_chunks == 0 || chunk_len == 0) return RR_OK;
    if (!host_in)
        return fail(RR_ERR_INVALID, shared ? "rr_chain_push_shared: host_in is null" : (summed ? "rr_chain_push_summed: host_in is null" : "rr_chain_push: host_in is null"));
    RR_CUDA(cudaSetDevice(c->ctx->device));
    const size_t len = chunk_len * n_chunks;
    const size_t S = (size_t)c->S;
    if (!shared && S > 1 && in_stride < len) return fail(RR_ERR_INVALID, "in_stride smaller than the pushed samples");
    // everything that can be refused is refused before anything is enqueued or any state advances
    Shape sh_in, sh_out;
    sh_in.chunk_len = chunk_len;
    sh_in.n_chunks = n_chunks;
    sh_in.rate = sample_rate;
    RR_TRY(dry_shape(c, sh_in, &sh_out));
    const size_t max_out = sh_out.len();
    if (max_out > out_capacity) return fail(RR_ERR_CAPACITY, "output buffer too small for this push");
    if (max_out > 0 && !host_out) return fail(RR_ERR_INVALID, summed ? "rr_chain_push_summed: host_out is null" : "rr_chain_push: host_out is null");
    if (!summed && max_out > out_stride && S > 1) return fail(RR_ERR_INVALID, "out_stride smaller than the produced samples");
    const size_t out_rows = summed ? 1 : S;
    if (!c->h2d_stream) {
        RR_CUDA(cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
        RR_CUDA(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            RR_CUDA(cudaEventCreateWithFlags(&c->ev_h2d[k], cudaEventDisableTiming));
            RR_CUDA(cudaEventCreateWithFlags(&c->ev_comp[k], cudaEventDisableTiming));
            RR_CUDA(cudaEventCreateWithFlags(&c->ev_d2h[k], cudaEventDisableTiming));
        }
    }
    const int b = c->slot;
    const size_t ocap = max_out ? max_out : 1;
    // (a staging buffer that has to grow is freed first: cudaFree waits for the work that still uses it)
    const size_t in_rows = shared ? 1 : S;
    RR_TRY(c->stage_in[b].ensure(in_rows * len * c->esz));
    RR_TRY(c->stage_out[b].ensure(out_rows * ocap * c->esz));
    // H2D of this push: behind the kernels of the push before last, which read the same slot
    RR_CUDA(cudaStreamWaitEvent(c->h2d_stream, c->ev_comp[b], 0));
    if (in_rows == 1 || in_stride == len)  // contiguous: one linear copy
        RR_CUDA(cudaMemcpyAsync(c->stage_in[b].p, host_in, in_rows * len * c->esz, cudaMemcpyHostToDevice, c->h2d_stream));
    else
        RR_CUDA(cudaMemcpy2DAsync(c->stage_in[b].p, len * c->esz, host_in, in_stride * c->esz, len * c->esz, S, cudaMemcpyHostToDevice,
                                  c->h2d_stream));
    RR_CUDA(cudaEventRecord(c->ev_h2d[b], c->h2d_stream));
    // kernels: behind that copy and behind the D2H copy that still reads this slot's output
    RR_CUDA(cudaStreamWaitEvent(c->stream, c->ev_h2d[b], 0));
    RR_CUDA(cudaStreamWaitEvent(c->stream, c->ev_d2h[b], 0));
    size_t produced = 0;
    RR_TRY(push_device(c, sample_rate, chunk_len, n_chunks, c->stage_in[b].p, len, shared, summed, c->stage_out[b].p, max_out, ocap,
                       &produced, out_sample_rate));
    RR_CUDA(cudaEventRecord(c->ev_comp[b], c->stream));
    if (produced > 0) {
        RR_CUDA(cudaStreamWaitEvent(c->d2h_stream, c->ev_comp[b], 0));
        if ((out_stride == ocap && produced == ocap) || out_rows == 1)
            RR_CUDA(cudaMemcpyAsync(host_out, c->stage_out[b].p, (out_rows == 1 ? produced : S * ocap) * c->esz, cudaMemcpyDeviceToHost,
                                    c->d2h_stream));
        else
            RR_CUDA(cudaMemcpy2DAsync(host_out, out_stride * c->esz, c->stage_out[b].p, ocap * c->esz, produced * c->esz, S,
                                      cudaMemcpyDeviceToHost, c->d2h_stream));
        RR_CUDA(cudaEventRecord(c->ev_d2h[b], c->d2h_stream));
    }
    c->slot ^= 1;
    if (out_count) *out_count = produced;
    return RR_OK;
}

}  // namespace

extern "C" {

int rr_chain_push_device(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in, size_t in_stride,
                         void* dev_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate) {
    return push_device(c, sample_rate, chunk_len, n_chunks, dev_in, in_stride, false, false, dev_out, out_capacity, out_stride, out_count,
                       out_sample_rate);
}

int rr_chain_push_shared_device(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in, void* dev_out,
                                size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate) {
    return push_device(c, sample_rate, chunk_len, n_chunks, dev_in, 0, true, false, dev_out, out_capacity, out_stride, out_count,
                       out_sample_rate);
}

int rr_chain_push(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* host_in, size_t in_stride,
                  void* host_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate) {
    return push_host(c, sample_rate, chunk_len, n_chunks, host_in, in_stride, false, false, host_out, out_capacity, out_stride, out_count,
                     out_sample_rate);
}

int rr_chain_push_shared(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* host_in, void* host_out,
                         size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate) {
    return push_host(c, sample_rate, chunk_len, n_chunks, host_in, 0, true, false, host_out, out_capacity, out_stride, out_count,
                     out_sample_rate);
}

int rr_chain_push_summed(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* host_in, size_t in_stride,
                         void* host_out, size_t out_capacity, size_t* out_count, double* out_sample_rate) {
    return push_host(c, sample_rate, chunk_len, n_chunks, host_in, in_stride, false, true, host_out, out_capacity, out_capacity, out_count,
                     out_sample_rate);
}

int rr_chain_push_summed_device(rr_chain* c, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in, size_t in_stride,
                                void* dev_out, size_t out_capacity, size_t* out_count, double* out_sample_rate) {
    return push_device(c, sample_rate, chunk_len, n_chunks, dev_in, in_stride, false, true, dev_out, out_capacity, out_capacity, out_count,
                       out_sample_rate);
}

// Device-to-device copy of `n_samples` samples per stream on the chain's copy stream (copy engine, no SM), ordered
// behind everything queued on the chain so far: moves a push's outputs into a buffer of another GPU (rr_ipc_open)
// while the next push computes.  The caller keeps `src_dev` untouched until the copy has run (two output buffers).
int rr_chain_copy_out_async(rr_chain* c, void* dst_dev, size_t dst_stride, const void* src_dev, size_t src_stride, size_t n_samples) {
    if (!c || (!dst_dev && n_samples) || (!src_dev && n_samples)) return fail(RR_ERR_INVALID, "rr_chain_copy_out_async: null argument");
    if (n_samples == 0) return RR_OK;
    RR_CUDA(cudaSetDevice(c->ctx->device));
    if (!c->d2h_stream) {
        RR_CUDA(cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
        RR_CUDA(cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            RR_CUDA(cudaEventCreateWithFlags(&c->ev_h2d[k], cudaEventDisableTiming));
            RR_CUDA(cudaEventCreateWithFlags(&c->ev_comp[k], cudaEventDisableTiming));
            RR_CUDA(cudaEventCreateWithFlags(&c->ev_d2h[k], cudaEventDisableTiming));
        }
    }
    if (!c->ev_copy) RR_CUDA(cudaEventCreateWithFlags(&c->ev_copy, cudaEventDisableTiming));
    RR_CUDA(cudaEventRecord(c->ev_copy, c->stream));
    RR_CUDA(cudaStreamWaitEvent(c->d2h_stream, c->ev_copy, 0));
    RR_CUDA(cudaMemcpy2DAsync(dst_dev, dst_stride * c->esz, src_dev, src_stride * c->esz, n_samples * c->esz, (size_t)c->S, cudaMemcpyDeviceToDevice,
                              c->d2h_stream));
    return RR_OK;
}

int rr_chain_sync(rr_chain* c) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    RR_CUDA(cudaSetDevice(c->ctx->device));
    RR_CUDA(cudaStreamSynchronize(c->stream));
    if (c->d2h_stream) RR_CUDA(cudaStreamSynchronize(c->d2h_stream));
    if (c->h2d_stream) RR_CUDA(cudaStreamSynchronize(c->h2d_stream));
    return RR_OK;
}
int rr_chain_set_fast_path(rr_chain* c, int enable) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    c->allow_poly = enable != 0;
    return RR_OK;
}
int rr_chain_set_timing(rr_chain* c, int enable) {
    if (!c) return fail(RR_ERR_INVALID, "null chain");
    RR_CUDA(cudaSetDevice(c->ctx->device));
    c->timing = enable != 0;
    c->ev_used = 0;
    return RR_OK;
}
int rr_chain_kernel_time(rr_chain* c, double* total_ms, int* n_launches, const char** kernel_name) {
    if (!c || !total_ms) return fail(RR_ERR_INVALID, "null argument");
    RR_CUDA(cudaSetDevice(c->ctx->device));
    // per kernel name: total and count; the dominant kernel (largest total) is reported here, the whole
    // list by rr_chain_kernel_breakdown
    std::vector<std::string> names;
    std::vector<double> tot;
    std::vector<int> cnt;
    for (size_t i = 0; i + 1 < c->ev_used; i += 2) {
        float ms = 0.f;
        RR_CUDA(cudaEventSynchronize(c->evs[i + 1]));
        RR_CUDA(cudaEventElapsedTime(&ms, c->evs[i], c->evs[i + 1]));
        const std::string& nm = c->ev_names[i / 2];
        size_t k = 0;
        while (k < names.size() && names[k] != nm) ++k;
        if (k == names.size()) {
            names.push_back(nm);
            tot.push_back(0.0);
            cnt.push_back(0);
        }
        tot[k] += ms;
        cnt[k] += 1;
    }
    size_t best = 0;
    c->breakdown.clear();
    for (size_t k = 0; k < names.size(); ++k) {
        if (tot[k] > tot[best]) best = k;
        char buf[160];
        std::snprintf(buf, sizeof buf, "%s%s:%.6f:%d", k ? ";" : "", names[k].c_str(), tot[k], cnt[k]);
        c->breakdown += buf;
    }
    *total_ms = names.empty() ? 0.0 : tot[best];
    if (n_launches) *n_launches = names.empty() ? 0 : cnt[best];
    c->timed_kernel = names.empty() ? "" : names[best];
    if (kernel_name) *kernel_name = c->timed_kernel.c_str();
    return RR_OK;
}
const char* rr_chain_kernel_breakdown(rr_chain* c) { return c ? c->breakdown.c_str() : ""; }
void* rr_chain_cuda_stream(rr_chain* c) { return c ? (void*)c->stream : nullptr; }
const char* rr_chain_plan(rr_chain* c) { return c ? c->plan.c_str() : ""; }

}  // extern "C"
