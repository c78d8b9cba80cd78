/* radiorust_b200 -- C ABI of the B200-native IQ sample chain.
 *
 * Drop-in boundary for ONE hot path of JanBeh/radiorust 0.5.0: the blocks
 * FreqShifter -> Filter -> Downsampler (+ Upsampler, FmDemod, de-emphasis,
 * GainControl).  The reference has no FFI of its own (pure Rust, SURVEY.md 8b);
 * these entry points are what an `extern "C"` FFI crate binds so that GPU
 * versions of the blocks can implement radiorust's Consumer/Producer traits
 * (src/flow.rs:233-267, src/blocks/mod.rs:111-144).  INTEGRATION.md shows the
 * Rust side.
 *
 * Conventions
 *  - plain C types, opaque handles, int status (0 = ok, < 0 = rr_status);
 *    rr_last_error() returns a THREAD-LOCAL message: read it on the thread that
 *    got the error code, before the next `.await` (Tokio tasks migrate between
 *    worker threads); nothing unwinds or aborts.
 *  - a push that is refused (RR_ERR_INVALID / UNSUPPORTED / CAPACITY) leaves the
 *    chain untouched.  A push that fails behind that check (RR_ERR_CUDA / NOMEM
 *    in mid-flight) resets the chain's streaming state: every block restarts as
 *    after rr_chain_create, parameters kept.
 *  - samples are interleaved complex (re, im): RR_C32 = num::Complex<f32>
 *    (8 bytes), RR_C64 = num::Complex<f64> (16 bytes) -- #[repr(C)] layout.
 *  - a chain processes `n_streams` independent streams in lock step; stream s
 *    lives at base + s*stride (stride in samples).
 *  - every call selects the handle's CUDA device first (Tokio tasks migrate
 *    between threads).  A handle is Send but not Sync: one task owns a chain.
 *  - there is NO CPU fallback: without a CUDA device rr_ctx_create fails.
 */
#ifndef RADIORUST_B200_H
#define RADIORUST_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RR_VERSION_MAJOR 0
#define RR_VERSION_MINOR 5

typedef struct rr_ctx rr_ctx;
typedef struct rr_chain rr_chain;
typedef struct rr_pool rr_pool;

typedef enum rr_status {
    RR_OK = 0,
    RR_ERR_INVALID = -1,     /* bad argument / contract violation (reference: assert!/panic in the task) */
    RR_ERR_CUDA = -2,        /* CUDA runtime error (message holds cudaGetErrorString) */
    RR_ERR_UNSUPPORTED = -3, /* valid for the reference, not implemented on the device path */
    RR_ERR_NOMEM = -4,
    RR_ERR_CAPACITY = -5     /* output buffer too small */
} rr_status;

typedef enum rr_dtype { RR_C32 = 0, RR_C64 = 1 } rr_dtype;

/* One stage = one reference block. */
typedef enum rr_stage_kind {
    RR_STAGE_FREQSHIFT = 1,  /* blocks::FreqShifter   src/blocks/transform.rs:266-391 */
    RR_STAGE_FILTER = 2,     /* blocks::filters::Filter src/blocks/filters.rs:110-298 */
    RR_STAGE_DOWNSAMPLE = 3, /* blocks::Downsampler   src/blocks/resampling.rs:14-146 */
    RR_STAGE_UPSAMPLE = 4,   /* blocks::Upsampler     src/blocks/resampling.rs:149-280 */
    RR_STAGE_FMDEMOD = 5,    /* blocks::modulation::FmDemod src/blocks/modulation.rs:83-158 */
    RR_STAGE_GAIN = 6,       /* blocks::GainControl   src/blocks/transform.rs:29-92 */
    RR_STAGE_FOURIER = 7,    /* blocks::analysis::Fourier src/blocks/analysis.rs:15-132 */
    RR_STAGE_FMMOD = 8,      /* blocks::modulation::FmMod src/blocks/modulation.rs:13-80 */
    RR_STAGE_RECHUNK = 9,    /* blocks::chunks::Rechunker src/blocks/chunks.rs:42-176 */
    RR_STAGE_OVERLAP = 10    /* blocks::chunks::Overlapper src/blocks/chunks.rs:179-248 */
} rr_stage_kind;

typedef enum rr_window_kind {
    RR_WINDOW_KAISER = 0,      /* windowing::Kaiser{beta}  src/windowing.rs:24-51 */
    RR_WINDOW_RECTANGULAR = 1, /* windowing::Rectangular   src/windowing.rs:14-20 */
    RR_WINDOW_CUSTOM = 2       /* windowing::CustomWindow  src/windowing.rs:58-67 */
} rr_window_kind;

/* Frequency response closure of Filter (`Fn(isize, f64) -> Complex<f64>`,
 * src/blocks/filters.rs:128-131): called on the host at (re)design time only. */
typedef void (*rr_freq_resp_fn)(void* user, int64_t bin, double freq_hz, double* out_re, double* out_im);
/* Window::relative_value_at (src/windowing.rs:9), x in [-1, 1]. */
typedef double (*rr_window_fn)(void* user, double x);

typedef struct rr_stage_desc {
    int32_t kind; /* rr_stage_kind */
    int32_t window_kind; /* FILTER: rr_window_kind */
    /* FREQSHIFT: FreqShifter::with_precision_and_shift(precision, shift) */
    double precision; /* hertz, reference default 1.0 */
    double shift;     /* hertz, initial value for every stream */
    /* FILTER: Filter::with_window(freq_resp, window) */
    rr_freq_resp_fn freq_resp;
    void* freq_resp_user;
    double window_beta; /* Kaiser beta; Filter::new uses sqrt(3) (= with_null_at_bin(2.0)) */
    rr_window_fn window_fn;
    void* window_user;
    /* DOWNSAMPLE / UPSAMPLE: ::with_quality(output_chunk_len, output_rate, bandwidth, quality) */
    uint64_t output_chunk_len;
    double output_rate;
    double bandwidth;
    double quality; /* reference default 3.0 */
    /* FMDEMOD: FmDemod::new(deviation) */
    double deviation;
    /* GAIN: GainControl::new(gain) */
    double gain;
    /* FOURIER: Fourier::with_window(window) / with_window_center_dc(window) (analysis.rs:38-59): window_kind,
     * window_beta, window_fn as for FILTER (RR_WINDOW_RECTANGULAR = Fourier::new); center_dc != 0 rotates the
     * DC bin to index n/2 (analysis.rs:113-115).  Output chunks have the input's length and sample rate. */
    int32_t center_dc;
    /* OVERLAP: Overlapper::new(chunk_count) (chunks.rs:194-196), > 0.  Output chunk = the last chunk_count input
     * chunks concatenated; nothing is emitted until chunk_count chunks have arrived.  The chunks of one history
     * must share length and sample rate (anything else returns RR_ERR_UNSUPPORTED and leaves the state alone). */
    int32_t chunk_count;
    /* FMMOD: FmMod::new(deviation) uses `deviation` above (modulation.rs:27).  The phase accumulator follows the
     * reference's rounding step by step (product, sum, fmod in Flt; modulation.rs:46-51) and survives events.
     * RECHUNK: Rechunker::new(output_chunk_len) uses `output_chunk_len` above (chunks.rs:57), > 0. */
} rr_stage_desc;

typedef struct rr_chain_desc {
    int32_t dtype;     /* rr_dtype */
    int32_t n_streams; /* independent streams processed per push */
    int32_t n_stages;
    int32_t reserved;
    const rr_stage_desc* stages;
} rr_chain_desc;

/* ---- library / errors ---------------------------------------------------- */
const char* rr_last_error(void);
int rr_version(int* major, int* minor);
/* number of kernels this library has launched in the calling process */
uint64_t rr_kernel_launch_count(void);

/* ---- context (one per device) -------------------------------------------- */
int rr_ctx_create(int device, rr_ctx** out);
int rr_ctx_destroy(rr_ctx* ctx);
int rr_ctx_device(const rr_ctx* ctx);

/* ---- pinned chunk pool at the chain edges (replaces bufferpool.rs:187-222) ---
 * ChunkBufPool for page-locked memory.  rr_pool_get = ChunkBufPool::get_with_capacity (bufferpool.rs:210-222): the
 * OLDEST recycled buffer is handed out again when it holds min_bytes (a smaller one is replaced: a Vec would grow in
 * place, pinned memory cannot), otherwise a new one is allocated; *capacity = its size.  rr_pool_put is the recycler
 * (Chunk::drop, bufferpool.rs:82-90): call it when the last owner of the chunk lets go.  get/put may come from any
 * thread (the reference's recycler is an mpsc channel).  rr_pool_destroy frees idle buffers and those still on loan. */
int rr_pool_create(rr_ctx* ctx, rr_pool** out);
int rr_pool_destroy(rr_pool* pool);
int rr_pool_get(rr_pool* pool, size_t min_bytes, void** out, size_t* capacity);
int rr_pool_put(rr_pool* pool, void* p);
int rr_pool_trim(rr_pool* pool); /* free the idle buffers */
int rr_pool_stats(rr_pool* pool, uint64_t* allocated, uint64_t* reused, uint64_t* idle_buffers, uint64_t* live_buffers);
/* one-off pinned allocations and in-place pinning of a recycled Vec (bufferpool.rs:202-222 reuses its Vecs, so a
 * registration amortises) */
int rr_pinned_alloc(rr_ctx* ctx, size_t bytes, void** out);
int rr_pinned_free(rr_ctx* ctx, void* p);
int rr_host_register(rr_ctx* ctx, void* p, size_t bytes);
int rr_host_unregister(rr_ctx* ctx, void* p);
int rr_device_alloc(rr_ctx* ctx, size_t bytes, void** out);
int rr_device_free(rr_ctx* ctx, void* p);
/* A device buffer of ANOTHER process's GPU (one process per GPU) as a local pointer: the owner exports a 64-byte
 * handle of a buffer it got from rr_device_alloc, the others open it (peer access over NVLink is enabled on
 * opening).  Passed as `dev_out` of rr_chain_push_device it makes the chain's last kernel store its outputs
 * straight into the owner's memory -- the gather of a channelizer's outputs (SURVEY.md 8e) without a collective
 * kernel.  The owner keeps the buffer allocated until every opener has closed it. */
int rr_ipc_export(rr_ctx* ctx, void* dev_ptr, void* handle_out_64_bytes);
int rr_ipc_open(rr_ctx* ctx, const void* handle_64_bytes, void** dev_ptr);
int rr_ipc_close(rr_ctx* ctx, void* dev_ptr);
/* synchronous copies; both first wait for ALL work queued on the device (chains run on their own non-blocking
 * streams), so they are safe right behind rr_chain_push_device without an rr_chain_sync */
int rr_memcpy_h2d(rr_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes);
int rr_memcpy_d2h(rr_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes);

/* ---- metering (src/metering.rs) ------------------------------------------
 * Synchronous; each call first waits for all work queued on the device, so the output of rr_chain_push_device can
 * be metered directly (no rr_chain_sync needed in between).  n_streams <= 65535. */
/* mean square norm of every chunk of DEVICE samples: host_out[s*n_chunks + c] for chunk c of stream s
 * (stream s at dev_in + s*in_stride samples); accumulated in f64 like the reference. */
int rr_metering_level(rr_ctx* ctx, int32_t dtype, const void* dev_in, size_t in_stride, size_t chunk_len, size_t n_chunks,
                      int n_streams, double* host_out);
/* metering::bandwidth (src/metering.rs:42-84) of every chunk of Fourier-transformed DEVICE samples (the output
 * of a FOURIER stage, DC at index 0): hertz that hold all but `double_percentile` of the energy,
 * host_out[s*n_chunks + c].  n_streams <= 65535. */
int rr_metering_bandwidth(rr_ctx* ctx, int32_t dtype, const void* dev_bins, size_t in_stride, size_t chunk_len, size_t n_chunks,
                          int n_streams, double double_percentile, double sample_rate, double* host_out);
/* metering::rescale_energy (src/metering.rs:93-110): `resolution` energies per chunk (Flt = float for RR_C32,
 * double for RR_C64), host_out[(s*n_chunks + c)*resolution + o]; expects DC in the centre (center_dc).
 * n_streams, n_chunks <= 65535. */
int rr_metering_rescale_energy(rr_ctx* ctx, int32_t dtype, const void* dev_bins, size_t in_stride, size_t chunk_len, size_t n_chunks,
                               int n_streams, size_t resolution, void* host_out);

/* ---- design math, host only (no GPU needed) ------------------------------ */
double rr_bessel_i0(double x);                      /* math::bessel_I0  src/math.rs:7-20 */
double rr_sinc(double x);                           /* math::sinc       src/math.rs:42-49 */
double rr_kaiser_rel_with_beta(double beta, double x); /* src/math.rs:26-28 */
double rr_kaiser_null_at_bin_to_beta(double n);     /* src/math.rs:37-39 */
void rr_deemphasis_factor(double tau, double frequency, double* out_re, double* out_im); /* filters.rs:20-27 */
int rr_freq_to_ratio(double sample_rate, double precision, double frequency, int64_t* numer, int64_t* denom); /* transform.rs:298-302 */
/* extended_response of Filter (2n complex f64 values, interleaved) -- filters.rs:184-238 */
int rr_design_filter_response(rr_freq_resp_fn f, void* f_user, int32_t window_kind, double window_beta,
                              rr_window_fn w, void* w_user, double sample_rate, size_t n, int32_t dtype,
                              double* out_2n_complex);
/* Downsampler / Upsampler taps; returns the tap count through *ir_len; pass ir == NULL to query */
int rr_design_downsampler_taps(double input_rate, double output_rate, double bandwidth, double quality,
                               size_t* ir_len, double* ir); /* resampling.rs:75-98 */
int rr_design_upsampler_taps(double input_rate, double output_rate, double bandwidth, double quality,
                             size_t* ir_len, double* ir);   /* resampling.rs:205-233 */

/* Diagnostic of the rank-reduced form of Filter -> Downsampler (in/out = P/Q reduced, Q <= 4): the P x (Lmax+1)
 * matrix of the fused filter g = taps(filters.rs:184-238) * reversed taps(resampling.rs:82-101) -- for Q > 1 the Q
 * phase matrices side by side -- is factored as sum_c a_c b_c^T; *rank = smallest count whose discarded part is
 * <= tol * |M|_F (0 if that needs more than max_rank), *discarded = that part, *table_error = relative L2 distance
 * between the factorisation and the full polyphase tables (K = 512). */
int rr_design_fused_rank(rr_freq_resp_fn f, void* f_user, int32_t window_kind, double window_beta, rr_window_fn w, void* w_user,
                         double sample_rate, size_t n, double output_rate, double bandwidth, double quality, double tol,
                         int max_rank, int* rank, double* discarded, double* table_error);

/* ---- chain ----------------------------------------------------------------- */
int rr_chain_create(rr_ctx* ctx, const rr_chain_desc* desc, rr_chain** out);
int rr_chain_destroy(rr_chain* chain);

/* FreqShifter::set_shift (transform.rs:384-386); stream < 0 = all streams.
 * Takes effect at the next push, phase-continuously (transform.rs:322-327). */
int rr_chain_set_shift(rr_chain* chain, int stage, int stream, double shift_hz);
/* one shift per stream in a single call (n must equal n_streams): a channelizer's tuning table */
int rr_chain_set_shifts(rr_chain* chain, int stage, const double* shifts_hz, int n);
/* FreqShifter::shift (transform.rs:380-382) */
int rr_chain_get_shift(rr_chain* chain, int stage, int stream, double* shift_hz);
/* Filter::update / update_with_window (filters.rs:279-297): redesign at the next
 * push and drop the history chunk (filters.rs:187). */
int rr_chain_update_filter(rr_chain* chain, int stage, rr_freq_resp_fn f, void* f_user, int32_t window_kind,
                           double window_beta, rr_window_fn w, void* w_user, int keep_window);
/* FmDemod::set_deviation (modulation.rs:154-157) / FmMod::set_deviation (modulation.rs:76-79) */
int rr_chain_set_deviation(rr_chain* chain, int stage, double deviation);
/* Rechunker::set_output_chunk_len (chunks.rs:171-175); takes effect with the next push */
int rr_chain_set_output_chunk_len(rr_chain* chain, int stage, size_t output_chunk_len);
/* GainControl::set (transform.rs:89-91) */
int rr_chain_set_gain(rr_chain* chain, int stage, double gain);

/* In-band event (signal.rs:19-31).  Interrupt events reset Filter history
 * (filters.rs:262-267) and FmDemod's previous sample (modulation.rs:133-138);
 * resamplers, FmMod and the NCO keep their state.  ANY event makes a Rechunker
 * drop its partial chunk (chunks.rs:84-91) and an Overlapper its history
 * (chunks.rs:226-233); each of them then sends `SamplesLost` (an interrupt,
 * chunks.rs:19-28) ahead of the event, so the stages behind it see an interrupt. */
int rr_chain_event(rr_chain* chain, int is_interrupt);
/* Number of `SamplesLost` events the chain's Rechunker / Overlapper stages have generated so far (on events, and
 * a Rechunker on a sample-rate change with a partial chunk pending, chunks.rs:71-79).  The block task compares the
 * count before and after rr_chain_event / a push and sends that many SamplesLost downstream first. */
uint64_t rr_chain_samples_lost_count(rr_chain* chain);

/* Upper bound of output samples per stream for a push of n_chunks*chunk_len
 * input samples at sample_rate. */
size_t rr_chain_max_output(rr_chain* chain, double sample_rate, size_t chunk_len, size_t n_chunks);

/* Signal::Samples{sample_rate, chunk} for every stream: `n_chunks` consecutive
 * chunks of `chunk_len` samples per stream (n_chunks > 1 batches several
 * reference messages into one launch; results are identical to pushing them one
 * by one).  HOST buffers (pinned for full asynchrony): H2D, kernels and D2H are
 * enqueued on the chain's stream; call rr_chain_sync before reading host_out.
 * *out_count = samples produced per stream (same for all streams);
 * *out_sample_rate = their rate.  out_count follows the reference: a Filter's
 * first chunk after start/redesign/interrupt only primes history
 * (filters.rs:240,260); resamplers emit whole chunks of output_chunk_len
 * (resampling.rs:121-131). */
int rr_chain_push(rr_chain* chain, double sample_rate, size_t chunk_len, size_t n_chunks, const void* host_in,
                  size_t in_stride, void* host_out, size_t out_capacity, size_t out_stride, size_t* out_count,
                  double* out_sample_rate);
/* Same with DEVICE buffers (no PCIe traffic; stays device-resident). */
int rr_chain_push_device(rr_chain* chain, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in,
                         size_t in_stride, void* dev_out, size_t out_capacity, size_t out_stride, size_t* out_count,
                         double* out_sample_rate);
/* Every stream reads the same n_chunks*chunk_len input samples (one row): a channelizer tuning all its streams
 * out of one wideband input.  Stream state (NCO phase, Filter history, resampler rings, ...) stays per stream;
 * outputs are laid out as for rr_chain_push[_device].  The results equal a push of the row replicated into
 * every stream, bit for bit, whenever both take the same plan.  The host form copies the row once (len samples,
 * not n_streams*len); the device form reads it in place, so its input costs no memory per stream.  Contract,
 * refusals and failure handling as for the per-stream pushes; the two kinds may be mixed on one chain. */
int rr_chain_push_shared(rr_chain* chain, double sample_rate, size_t chunk_len, size_t n_chunks, const void* host_in,
                         void* host_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate);
int rr_chain_push_shared_device(rr_chain* chain, double sample_rate, size_t chunk_len, size_t n_chunks, const void* dev_in,
                                void* dev_out, size_t out_capacity, size_t out_stride, size_t* out_count, double* out_sample_rate);
int rr_chain_sync(rr_chain* chain);
/* Copy `n_samples` samples per stream from one device buffer to another (a buffer of another GPU opened with rr_ipc_open,
 * for example) on the chain's copy stream -- a copy engine, no SM -- behind everything queued on the chain so far: a
 * push's outputs travel to the gathering GPU while the next push computes.  Keep src_dev untouched until the copy has
 * run (alternate between two output buffers); rr_chain_sync waits for it. */
int rr_chain_copy_out_async(rr_chain* chain, void* dst_dev, size_t dst_stride, const void* src_dev, size_t src_stride, size_t n_samples);
/* The fused Filter -> Downsampler kernels (rank-reduced front end + low-rate
 * polyphase part, or the polyphase kernels on all P branches) are used whenever
 * the chain allows it; enable = 0 forces the stateful overlap-save path (same
 * results within rounding; for tests and comparisons).  Env RR_DISABLE_POLY=1
 * sets the default to off; RR_DISABLE_FRONT=1 / RR_DISABLE_POLY2=1 step back to
 * k_poly2 on all branches / to k_poly (RR_DISABLE_FRONT also switches off the shared
 * front end of rates with several output phases).  Long Filters (2n = 2^15 .. 2^20):
 * RR_BIG_OS_LEGACY=1 keeps the round-1 four-step kernels. */
int rr_chain_set_fast_path(rr_chain* chain, int enable);
/* Measurement aid: while enabled, CUDA events on the chain's stream bracket the
 * dominant kernel of every push (no synchronisation is added).
 * rr_chain_kernel_time waits for the recorded pairs and returns, for the kernel
 * with the largest summed duration, that duration, its launch count and its
 * name; rr_chain_set_timing(.., 1) restarts the record. */
int rr_chain_set_timing(rr_chain* chain, int enable);
int rr_chain_kernel_time(rr_chain* chain, double* total_ms, int* n_launches, const char** kernel_name);
/* every timed kernel of the record as "name:total_ms:launches;..." (valid after rr_chain_kernel_time,
 * which reports the one with the largest total) */
const char* rr_chain_kernel_breakdown(rr_chain* chain);
/* raw cudaStream_t of the chain (for event timing by the caller) */
void* rr_chain_cuda_stream(rr_chain* chain);
/* name of the execution plan chosen at the last push (diagnostics), e.g.
 * "nco+fused[filter+down]" (k_fused), "nco+front+poly2[filter+down]" (k_front + k_poly2),
 * "nco+front+poly[filter+down]" (several output phases: k_front / k_front_wide + k_poly on u),
 * "fused_os[nco+filter+down]" or "big_os|fmdemod|front+poly[filter+down]" */
const char* rr_chain_plan(rr_chain* chain);

#ifdef __cplusplus
}
#endif
#endif /* RADIORUST_B200_H */
