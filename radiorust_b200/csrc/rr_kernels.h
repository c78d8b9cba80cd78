// Host-callable launchers of the sm_100a kernels (C++ linkage, internal to the
// library; the public boundary is include/radiorust_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rr {

// Per-stream NCO state (device resident).  Mirrors the task-local state of
// FreqShifter (src/blocks/transform.rs:307-309): the reduced ratio
// numer/denom, the start phase and the running table index.
struct NcoStream {
    uint32_t numer_abs;   // |numer| (< denom)
    uint32_t denom;       // > 0, < 2^31
    uint32_t idx;         // phase_idx, < denom
    int32_t sign;         // sign(numer): -1, 0, +1
    double start_phase;   // radians (value of Flt precision)
};

// Decimation geometry for integer-valued rates: in/out = P/Q reduced.
// j0 = input samples consumed so far (reduced mod P), m0 = outputs emitted so
// far (reduced consistently); output m fires at input count ceil(m*P/Q)
// (src/blocks/resampling.rs:109-111 in closed form).
struct RateState {
    long long P, Q, j0, m0;
};

template <typename T> struct ChainOsArgs {
    const void* in;         // [S][in_stride] complex<T>
    long long in_stride;    // elements
    int n_chunks;           // chunks in this launch (including a history-only first chunk)
    int first_is_history;   // 1: no stored history; chunk 0 only primes the filter
    int emit;               // 0: state-only run (no samples written, only hist/ztail state)
    int reserved;
    const void* hist_in;    // post-NCO history chunk of stream s at hist_in + s*hist_stride (read when !first_is_history)
    long long hist_stride;  // elements
    void* hist_out;         // [S][n] new history or nullptr (never aliases hist_in: CTAs of one launch read and write)
    const void* hperm;      // [N] complex<T>, H(f) in FftPlan::hperm_index order
    const void* twN;        // [N] complex<T>, exp(-j*2*pi*e/N)
    const NcoStream* nco;   // [S] or nullptr (read-only; the host advances idx with launch_nco_advance)
    long long nco_offset;   // samples between nco[s].idx and sample 0 of `in`
    void* out;              // [S][out_stride] complex<T>
    long long out_stride;
    // decimating epilogue (EPI == 1)
    const T* ir;            // [L]
    int L;
    const void* ztail_in;   // [S][L-1] complex<T>: filter output preceding this launch
    void* ztail_out;        // [S][L-1]
    RateState rate;
};

// n = chunk length (N = 2n).  epi: 0 = write the filter output, 1 = decimating FIR.
// parts > 1 (EPI == 0 only) splits the chunks of every stream over `parts` CTAs.
template <typename T>
cudaError_t launch_chain_os(int n, int epi, int n_streams, int parts, const ChainOsArgs<T>& a, cudaStream_t st);
// true when (T, n, epi, L) can run in the fused single-CTA kernel
template <typename T> bool chain_os_supported(int n, int epi, int L);
template <typename T> int chain_os_threads(int n);
// index of true bin k in the permuted H table for chunk length n
template <typename T> int chain_os_hperm_index(int n, int k);

// ---- standalone stages ------------------------------------------------------
template <typename T>
cudaError_t launch_freqshift(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                             int n_streams, const NcoStream* nco, long long nco_offset, cudaStream_t st);

cudaError_t launch_nco_advance(NcoStream* nco, int n_streams, long long len, cudaStream_t st);

template <typename T>
cudaError_t launch_gain(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                        int n_streams, double gain, cudaStream_t st);

// FIR decimator on [tail(L-1) | input(len)] (src/blocks/resampling.rs:103-121)
template <typename T>
cudaError_t launch_downsample(const void* in, long long in_stride, long long len, const void* tail_in, void* tail_out,
                              const T* ir, int L, RateState rate, long long n_out, void* out, long long out_stride,
                              int n_streams, cudaStream_t st);

// zero-stuffing interpolator, gather form (src/blocks/resampling.rs:238-267)
// out2 (optional; integer interpolation factors only, see upsample_tiled_supported): outputs o >= out_split go to
// out2[o - out_split] instead of out[o]
template <typename T>
cudaError_t launch_upsample(const void* in, long long in_stride, long long len, const void* acc_in, void* acc_out,
                            const T* ir, int L, RateState rate, long long n_out, void* out, long long out_stride,
                            int n_streams, cudaStream_t st, void* out2 = nullptr, long long out2_stride = 0, long long out_split = 0);
template <typename T> bool upsample_tiled_supported(RateState rate, int L);
// the integer factors that launch_upsample runs one output phase per thread (k_upsample_phase), taps in registers
inline bool upsample_phase_supported(RateState rate, int L, long long n_out) {
    return rate.P == 1 && rate.Q >= 8 && rate.Q <= 256 && L >= 1 && (L + rate.Q - 1) / rate.Q <= 16 && n_out + L < (1LL << 40);
}

// ---- summed-output pushes (rr_synth.cu) ---------------------------------------
// k_synth: the chain's last two stages Upsampler (upsample_phase_supported) -> FreqShifter of every stream, added into
// one row.  Row sample t of the push is the FreqShifter's output t of every stream: the samples pending in the
// Upsampler's staging buffer for t < pending, its new output o = t - pending behind them.
struct SynthArgs {
    const void* in;         // [S][in_stride] complex<T>: the Upsampler's input of this push
    long long in_stride, len;
    const void* acc_in;     // [S][L]: partial sums carried into this push
    void* acc_out;          // [S][L]: outputs o >= n_new, carried into the next push
    const void* ir;         // [L] T
    int L, Q;               // taps; in/out = 1/Q
    long long j0, m0;       // RateState of the push
    long long n_new;        // new Upsampler outputs per stream
    const void* pend;       // [S][obuf_stride]: samples pending before the push (pre-NCO)
    long long pending;
    void* rem;              // [S][obuf_stride]: outputs o >= split, the Upsampler's next pending part (pre-NCO)
    long long obuf_stride, split;
    const NcoStream* nco;   // [S] the FreqShifter's state at the push (read-only)
    void* out;              // the row: `emit` = pending + split samples
    long long emit;
};
template <typename T> cudaError_t launch_synth(const SynthArgs& a, int n_streams, int sm_count, cudaStream_t st);
// k_stream_sum: out[t] = sum over s ascending of in[s*in_stride + t], in f64 from +0.0, rounded once to T
template <typename T>
cudaError_t launch_stream_sum(const void* in, long long in_stride, long long len, int n_streams, void* out, cudaStream_t st);

// The resamplers with their firing pattern from tables (rates that are not integer valued; the tables replay the
// reference's f64 `pos` recurrence, resampling.rs:109-111 / :247-266): fire[o] = input sample of this push that output o
// ends at; qpos[p] = output cell input p starts at, cnt[i] = inputs with qpos <= i
template <typename T>
cudaError_t launch_downsample_indexed(const void* in, long long in_stride, long long len, const void* tail_in, void* tail_out, const T* ir, int L,
                                      const int* fire, long long n_out, void* out, long long out_stride, int n_streams, cudaStream_t st);
template <typename T>
cudaError_t launch_upsample_indexed(const void* in, long long in_stride, long long len, const void* acc_in, void* acc_out, const T* ir, int L,
                                    const int* qpos, const int* cnt, long long n_out, void* out, long long out_stride, int n_streams,
                                    cudaStream_t st);

// FM discriminator (src/blocks/modulation.rs:116-126)
template <typename T>
cudaError_t launch_fmdemod(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                           int n_streams, void* prev_sample, void* last_output, int has_prev, double factor,
                           cudaStream_t st);

// FmMod (src/blocks/modulation.rs:46-51): phase[s] is the accumulator carried across pushes (Flt)
template <typename T>
cudaError_t launch_fmmod(const void* in, long long in_stride, void* out, long long out_stride, long long len, int n_streams, void* phase,
                         double factor, int sm_count, cudaStream_t st);

// Overlapper gather (src/blocks/chunks.rs:203-225): out[j*span + t] = seq[base + j*hop + t], seq = a (a_len samples) | b
template <typename T>
cudaError_t launch_overlap(const void* a, long long a_stride, long long a_len, const void* b, long long b_stride, void* out,
                           long long out_stride, long long n_out, long long span, long long hop, long long base, int n_streams,
                           cudaStream_t st);

// Fourier analysis block (src/blocks/analysis.rs:60-132): out chunk = FFT_n(window * in chunk), bin k at
// (k + rot) mod n.  Three-pass FFT for the plan sizes, direct DFT for any other n <= kFourierDirectMax.
constexpr int kFourierDirectMax = 4096;
template <typename T> bool fourier_fft_supported(int n);
template <typename T>
cudaError_t launch_fourier(int n, const void* in, long long in_stride, void* out, long long out_stride, int n_chunks, int n_streams,
                           const T* window, const void* twN, int rot, cudaStream_t st);

// metering::level (src/metering.rs:21-30): out[s*n_chunks + c] = mean |x|^2 of chunk c of stream s (f64, device)
template <typename T>
cudaError_t launch_level(const void* in, long long in_stride, long long chunk_len, long long n_chunks, int n_streams, double* out,
                         cudaStream_t st);

// metering::bandwidth (src/metering.rs:42-84) of every chunk of Fourier-transformed samples: out[s*n_chunks + c] (f64, device)
template <typename T>
cudaError_t launch_bandwidth(const void* in, long long in_stride, long long chunk_len, long long n_chunks, int n_streams,
                             double double_percentile, double sample_rate, double* out, cudaStream_t st);
// metering::rescale_energy (src/metering.rs:93-110): out[(s*n_chunks + c)*resolution + o] (Flt, device)
template <typename T>
cudaError_t launch_rescale_energy(const void* in, long long in_stride, long long chunk_len, long long n_chunks, int n_streams,
                                  long long resolution, void* out, cudaStream_t st);

// strided 2-D copy of complex samples (used to stage stream buffers)
template <typename T>
cudaError_t launch_copy2d(const void* in, long long in_stride, void* out, long long out_stride, long long len,
                          int n_streams, cudaStream_t st);

// ---- large overlap-save (four-step FFT through L2-resident scratch) ---------
template <typename T> struct BigOsArgs {
    const void* in;         // [S][in_stride]: the pushed chunks
    long long in_stride;
    const void* hist;       // chunk preceding `in`, stream s at hist + s*hist_stride (read when block 0 starts at chunk 0)
    long long hist_stride;
    int first_chunk;        // block b convolves chunks (first_chunk + b - 1, first_chunk + b)
    int n_blocks;           // overlap-save blocks in this launch
    void* scratch;          // [S*n_blocks][N] complex<T>
    const void* hbig;       // [Na][Nb] H(f): row k1 holds bins k1 + Na*k2 in the row plan's hperm order
    const void* twN;        // [N] exp(-j*2*pi*e/N) (four-step twiddles)
    const void* twA;        // [Na] column-plan twiddles
    const void* twB;        // [Nb] row-plan twiddles
    void* out;              // [S][out_stride]
    long long out_stride;
    const void* twC;        // rr_long_os.cu: [long_os_twc_size] W_N^(long_os_twc_exponent(i)), the column tiles' twiddle factors
};
template <typename T> bool big_os_supported(int n);
template <typename T> void big_os_shape(int n, int* Na, int* Nb);
// position of true bin k in the permuted big-H table
template <typename T> long long big_os_hperm_index(int n, long long k);
template <typename T>
cudaError_t launch_big_os(int n, int n_streams, const BigOsArgs<T>& a, cudaStream_t st);
// 2n = 2^15 .. 2^20: three streaming kernels, N = Na x 1024 (rr_long_os.cu); the big_os_* entry points dispatch to them
bool long_os_supported(int n);
void long_os_shape(int n, int* Na, int* Nb);
long long long_os_hperm_index(int n, long long k);
template <typename T>
cudaError_t launch_long_os(int n, int n_streams, const BigOsArgs<T>& a, cudaStream_t st);
template <typename T> int long_os_twc_size(int n);
template <typename T> long long long_os_twc_exponent(int n, int i);

// ---- polyphase fused chain: NCO -> Filter -> Downsampler without the full-rate
// intermediate (rr_poly.cuh) ---------------------------------------------------
template <typename T> struct PolyArgs {
    const void* in;        // [S][in_stride] complex<T>: the pushed samples (pre-NCO)
    long long in_stride;
    long long len;         // pushed samples per stream
    const void* hist2;     // [S][2n] complex<T>: the 2n post-NCO samples preceding `in`
    long long n;           // Filter chunk length
    const NcoStream* nco;  // [S] or nullptr
    const void* gtab;      // [Q][P][K] complex<T>, bins in the K-point plan's hperm order
    const void* twK;       // [K] exp(-j*2*pi*e/K)
    long long P, Q;        // in/out = P/Q reduced
    int Lmax, V;           // low-rate filter reach, valid outputs per block and phase
    int n_blocks, nbpc;    // blocks per stream, blocks per CTA (k_poly2: per group)
    int ngrp;              // k_poly2: groups of nbpc blocks that one CTA half works through
    int halves;            // k_poly2: independent halves per CTA (0 or 2: two; 1: one half per CTA, half the shared memory)
    // k_poly2, optional second destination: outputs with index o = m - m0 - 1 >= out_split go to out2[o - out_split]
    // (the samples behind the last whole output chunk: the Downsampler's next pending part), the others to out[o]
    void* out2;
    long long out2_stride, out_split;  // out2 == nullptr: everything to `out`
    // k_poly2, streams as blocks (sab_blocks > 0; used when a stream has only sab_rb <= 3 blocks, i.e. short pushes): a
    // "stream" of this launch is a run of sab_blocks/sab_rb real streams; its block b is block b % sab_rb of real
    // stream s*(sab_blocks/sab_rb) + b/sab_rb -- window start (b/sab_rb)*sab_in_step + (b%sab_rb)*V*P, destinations
    // moved by (b/sab_rb)*sab_out_step (out) and *sab_out2_step (out2); real streams >= sab_streams do not exist.
    // One inverse round then serves up to nbpc blocks of several streams instead of one stream's few.
    int sab_blocks, sab_rb, sab_streams;
    long long sab_in_step, sab_out_step, sab_out2_step;
    long long J0, m0;      // filter-output samples consumed / outputs emitted before this push (reduced)
    long long m_lo, m_hi;  // outputs m to produce (inclusive)
    long long I_lo;        // low-rate index of block 0's first valid output
    void* out;             // [S][out_stride]; output m goes to out[m - m0 - 1]
    long long out_stride;
};
template <typename T> bool poly_supported(int K, int Q, int G);
template <typename T> int poly_hperm_index(int K, int k);
template <typename T> size_t poly_smem_bytes(int K, int Q, int G, int nbpc);
template <typename T> cudaError_t launch_poly(int K, int Q, int G, int n_streams, const PolyArgs<T>& a, cudaStream_t st);

// The pushed samples (len complex f32 per stream, n_streams rows in_stride apart; shared: one row that every stream
// reads) can be read through a TMA tensor map (rr_tma.cuh): 16-byte aligned base, rows a multiple of 16 bytes apart,
// fewer than 2^31 samples.  k_poly2, k_front and k_fused on the input need it; their launchers refuse what fails it.
inline bool tma_input_ok(const void* in, long long in_stride, long long len, int n_streams, bool shared) {
    return ((uintptr_t)in % 16 == 0) && (n_streams == 1 || shared || in_stride % 2 == 0) && len < (1LL << 31);
}

// ---- k_poly2 (rr_poly2.cu): the complex-f32, Q == 1 form of the polyphase chain on packed
// fp32 instructions with TMA-fed tiles.  Same PolyArgs; `gtab` is laid out by poly2_table_index.
bool poly2_supported(int K, long long P, long long Q);
int poly2_pick_G(long long P);
size_t poly2_smem_bytes(int G, int nbpc);
// position (complex elements) of bin k of branch p = r*G + g in the device table
long long poly2_table_index(int G, int r, int g, int k);
// shared_in: every stream reads the one row at a.in (a.in_stride == 0, n_streams > 1); a zero stride without it is refused
cudaError_t launch_poly2(int G, int n_streams, const PolyArgs<float>& a, bool shared_in, int sm_count, cudaStream_t st);

// ---- k_front (rr_front.cu): rank-reduced front end u_c[i] = sum_p a_c[p] * x'[i*P + p] (f32, Q == 1).
// k_poly2 then runs on u as a stream of `rank_pad` branches.
struct FrontArgs {
    const void* in;        // [S][in_stride] complex<float>: the pushed samples (pre-NCO)
    long long in_stride;
    long long len;         // pushed samples per stream
    const void* hist2;     // [S][2n]: the 2n post-NCO samples preceding `in`
    long long n;
    const NcoStream* nco;  // [S] or nullptr
    const float* acoef;    // [P/2][2][rank_pad]: a_c[p] at ((p/2)*2 + (p&1))*rank_pad + c
    int P;
    long long J0;          // as PolyArgs::J0: row r, branch p is push sample r*P + p - J0
    long long row_first;   // row index of u row 0
    int n_rows;            // rows to produce per stream
    void* u;               // [S][u_stride] complex<float>, row-major [row][rank_pad]
    long long u_stride;    // complex elements, even
    int tiles_per_warp;    // set by the launcher
    int has_hist_map;      // set by the launcher: history tiles come by TMA from hist2
    // optional: the mixed samples at push offsets >= hist_from also go to hist_out[s][offset - hist_from]
    // (the Filter's next history, [S][hist_stride]), for every offset inside the rows this launch covers
    void* hist_out;
    long long hist_from, hist_stride;
    int hist_staged;       // != 0: history samples go through the shared-memory tile (coalesced stores)
    // optional: kept_rows rows of u computed by the previous push ([S][kept_stride] complex, rows of rank_pad) are copied
    // to the kept_rows rows in front of `u` (the history rows of this push)
    const void* kept_src;
    long long kept_stride;
    int kept_rows;
};
bool front_supported(int rank_pad, long long P);
cudaError_t launch_front(int rank_pad, int n_streams, const FrontArgs& a, bool shared_in, int sm_count, cudaStream_t st);  // shared_in: as launch_poly2
// k_front_wide (rr_front_wide.cu): the same front end for any P (odd, thousands), 16 or 32 columns; `acoef` is
// [P][rank_pad]; kept rows are not taken
bool front_wide_supported(int rank_pad, long long P);
cudaError_t launch_front_wide(int rank_pad, int n_streams, const FrontArgs& a, cudaStream_t st);

// ---- k_fused (rr_fused.cu): front end + low-rate part in one persistent kernel; u stays in shared memory.
// Rows are numbered from the push's first new row: row r, column p is push sample r*P + p - J0, output r = row r's.
struct FusedArgs {
    const void* in;        // [S][in_stride] complex<float>: the pushed samples (pre-NCO)
    long long in_stride;
    long long len;
    const void* hist2;     // [S][2n]: the 2n post-NCO samples preceding `in` (row 0 may reach into them)
    long long n;
    const NcoStream* nco;  // [S] or nullptr
    int P;
    int coef_slot;         // constant-memory slot holding acoef ([P/2][2][10], as FrontArgs::acoef)
    int coef_off4;         // set by the launcher
    long long J0;          // 0 <= J0 < P
    int n_out;             // new rows (= outputs) per stream, >= 1
    int Lmax, V;           // reach of the low-rate filter, new rows per block (511 - Lmax)
    const void* ukeep_in;  // [S][ukeep_in_stride] complex: the Lmax rows of u preceding row 0, rows of 10
    long long ukeep_in_stride;
    void* ukeep_out;       // [S][ukeep_out_stride]: the last Lmax rows of this push
    long long ukeep_out_stride;
    const void* gtab;      // FFT_512(b_c) in poly2_table_index(10, 0, c, k) order
    const void* twK;       // [512] exp(-j*2*pi*e/512)
    void* out;             // [S][out_stride]; output o to out[o], or to out2[o - out_split] when o >= out_split
    long long out_stride;
    void* out2;
    long long out2_stride, out_split;
    // optional: the mixed samples at push offsets >= hist_from also go to hist_out[s][offset - hist_from]
    void* hist_out;
    long long hist_from, hist_stride;
};
bool fused_supported(int rank_pad, long long P, int Lmax);
int fused_coef_slots();
cudaError_t fused_upload_coef(int slot, const float* acoef, int P, cudaStream_t st);  // acoef: device memory, as FrontArgs::acoef
cudaError_t launch_fused(int n_streams, const FusedArgs& a, bool shared_in, int sm_count, cudaStream_t st);  // shared_in: as launch_poly2

// new hist2 = last 2n post-NCO samples of [hist2_in | in]; only entries [j_lo, j_hi) (j_hi < 0: 2n) -- the
// others were written by k_front
template <typename T>
cudaError_t launch_hist2_update(const void* in, long long in_stride, long long len, const void* hist2_in, void* hist2_out,
                                long long n, const NcoStream* nco, int n_streams, cudaStream_t st, long long j_lo = 0, long long j_hi = -1);

}  // namespace rr
