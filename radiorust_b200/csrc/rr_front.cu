// k_front: rank-reduced front end of the fused chain FreqShifter -> Filter ->
// Downsampler for integer decimation P (rr_design.h: design_rank_tables).
//
// The fused filter of the chain is y_m = sum_l sum_p M[p][l] x'[(m-1-l)P + p]
// (x' = NCO-mixed input, M[p][l] = g[P-1-p + lP], g = Filter taps * reversed
// Downsampler taps).  M = sum_c a_c b_c^T with `RK` real orthonormal a_c to
// below f32 rounding, so
//     u_c[i] = sum_p a_c[p] * x'[iP + p]                 (this kernel)
//     y      = sum_c (b_c * u_c)   at the output rate     (k_poly2 on u, RK branches)
// Every input sample is read once, mixed once (one complex multiply) and feeds
// RK real multiply-adds on the two-wide fp32 pipe; nothing of size P*K is ever
// transformed.  This is the HBM-bound half of the path: 8 B read and 8*RK/P B
// written per input sample.
//
// A warp takes 16 consecutive rows (= 16*P consecutive samples of one stream,
// one TMA box) into its own two-slot ring of shared-memory tiles; a lane pair
// per row, each lane half of the row's columns, the two partial results meet in
// one shuffle per result.  With P/2 odd the 16-byte loads of lanes that sit P*8
// bytes apart are conflict free.  16 warps per SM, each with a tile in flight
// while it works on the other.  The
// NCO phasor of sample (i, p) factors into the row phasor (exact per row from
// the integer phase recurrence, transform.rs:333-338, applied to the RK results
// of the row) and exp(j*w*p) (a P-entry table, applied to the sample).
// Rows that reach before the pushed samples (hist2: already mixed) or past them
// are loaded by their lane from global memory instead.
//
// Reference semantics: transform.rs:333-348 (NCO), filters.rs:240-253,
// resampling.rs:103-121.
#include <cuda.h>
#include <cuda_runtime.h>

#include <mutex>
#include <type_traits>

#include "rr_kernels.h"
#include "rr_poly.cuh"
#include "rr_pk.cuh"

namespace rr {

namespace {

constexpr int FR_WARPS = 4;
constexpr int FR_ROWS = 16;  // rows per tile: a lane pair per row, each lane half of the columns
constexpr int FR_STAGES = 2;  // tiles per warp in shared memory (one being filled while the other is used)
// bytes between the coefficient rows of consecutive steps ([2][RK] floats each).  The two lanes of a pair read rows that
// lie a multiple of four steps apart: sixteen columns (128-byte rows) get one 16-byte unit of padding, so that those rows
// start on different banks
constexpr int front_coef_pitch(int rk) { return 2 * rk * 4 + ((2 * rk * 4) % 128 == 0 ? 16 : 0); }

__device__ __forceinline__ uint32_t f_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ pc lds_front(uint32_t addr) {
    pc r;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(addr));
    return r;
}

// SHARED_IN: every stream reads the same input row (the input map holds that one row; the history map stays per stream)
template <int RK, bool HAS_NCO, bool SHARED_IN>
__global__ void __launch_bounds__(FR_WARPS * 32, 4) k_front(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_h, const FrontArgs a) {
    static_assert(RK == 10 || RK == 16, "results leave as 16-byte pairs: 6 + 4 per lane pair for ten columns, 8 + 8 for sixteen");
    constexpr int RK_SPLIT = RK == 10 ? 6 : RK / 2;  // lane hh = 0 stores results [0, RK_SPLIT), lane hh = 1 the rest
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = lane >> 1, hh = lane & 1;  // row of the tile, half of its columns
    const int s = blockIdx.y;
    const int P = a.P;
    const int steps = P / 2;
    // tile row pitch in samples: P, or P + 2 when P/2 is even (an odd number of 16-byte units per row keeps the
    // lanes' 16-byte loads conflict free); the two extra samples of a row are never used
    const int pitch = P + ((P & 3) == 0 ? 2 : 0);
    // Column pairs of this lane: [st0, st1).  An odd number of pairs (P = 2 mod 4) is split evenly and the last
    // pair is shared, one sample per lane.  The split point: with an odd number of 16-byte units per row the 8
    // lanes of a quarter warp (4 rows x 2 halves) hit 8 distinct bank groups when the halves start 4 (mod 8)
    // units apart.
    const bool odd_steps = (steps & 1) != 0;
    const int full = steps - (odd_steps ? 1 : 0);
    int split = full / 2;
    if (!odd_steps && steps >= 20) {
        for (int d = -1; d <= 1; ++d)
            if (((full / 2 + d) & 7) == 4) split = full / 2 + d;
    }
    const int st0 = hh ? split : 0, st1 = hh ? full : split;
    // lane hh = 1 walks its steps from `rot` on and wraps round: at any moment its 16-byte unit of the row (and its
    // coefficient row) lies split + rot = 4 (mod 8) units from its partner's, whatever the split -- the two halves of a
    // quarter warp then never meet on a bank.  (The sums are taken in another order than with rot = 0; still one fixed order.)
    const int cnt = st1 - st0;
    const int rot = (hh && cnt > 0) ? ((4 - (split & 7)) & 7) % cnt : 0;
    constexpr int CP = front_coef_pitch(RK);

    extern __shared__ __align__(128) unsigned char smem[];
    const int tile_bytes = FR_ROWS * pitch * 8;
    const int tile_stride = (tile_bytes + 127) / 128 * 128;
    unsigned char* tiles = smem + warp * (FR_STAGES * tile_stride);          // this warp's ring of tiles
    float* coef = reinterpret_cast<float*>(smem + FR_WARPS * FR_STAGES * tile_stride);  // [steps][2][RK]
    float2* colph = reinterpret_cast<float2*>(coef + (steps + 1) * (CP / 4));  // [P]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(colph + P);
    const uint32_t bar0 = f_smem_u32(&bars[warp * FR_STAGES]);

    uint32_t denom = 1, numer_abs = 0, idx0 = 0;
    int sign = 0;
    float start = 0.f;
    if (HAS_NCO) {
        const NcoStream ns = a.nco[s];
        denom = ns.denom;
        numer_abs = ns.numer_abs;
        sign = ns.sign;
        idx0 = ns.idx;
        start = (float)ns.start_phase;
    }
    for (int e = threadIdx.x; e < P * RK; e += FR_WARPS * 32) coef[(e / (2 * RK)) * (CP / 4) + e % (2 * RK)] = a.acoef[e];
    for (int p = threadIdx.x; p < P; p += FR_WARPS * 32) {
        cx<float> r(1.f, 0.f);
        if (HAS_NCO) r = nco_rotation<float>(p, numer_abs, denom, sign);
        colph[p] = make_float2(r.x, r.y);
    }
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < FR_STAGES; ++q) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + q * 8) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const float2* __restrict__ in = reinterpret_cast<const float2*>(a.in) + (long long)s * a.in_stride;
    const float2* __restrict__ hist_end = reinterpret_cast<const float2*>(a.hist2) + ((long long)s + 1) * 2 * a.n;
    float4* __restrict__ u = reinterpret_cast<float4*>(reinterpret_cast<float2*>(a.u) + (long long)s * a.u_stride);
    const long long len = a.len, hist_len = 2 * a.n;
    const long long hist_cap = len - a.hist_from;  // entries of hist_out that exist: push offsets below len
    float2* __restrict__ hist_o = a.hist_out ? reinterpret_cast<float2*>(a.hist_out) + (long long)s * a.hist_stride : nullptr;
    const uint32_t tiles_s = f_smem_u32(tiles);
    const uint32_t coef_s = f_smem_u32(coef), col_s = f_smem_u32(colph);

    // rotation of the row phasor from one tile to the next
    pc rot_tile(1.f, 0.f);
    if (HAS_NCO) {
        const cx<float> r = nco_rotation<float>((long long)FR_ROWS * P, numer_abs, denom, sign);
        rot_tile = pc(r.x, r.y);
    }

    const int tile0 = (blockIdx.x * FR_WARPS + warp) * a.tiles_per_warp;
    const int n_tiles = min(a.tiles_per_warp, (a.n_rows - tile0 * FR_ROWS + FR_ROWS - 1) / FR_ROWS);  // may be <= 0
    // push offset of the first sample of this warp's tile k (the launcher guarantees that offsets fit 32 bits)
    const int pos_first = (int)(((long long)a.row_first + (long long)tile0 * FR_ROWS) * P - a.J0), pos_step = FR_ROWS * P;
    const int len32 = (int)len;
    auto tile_pos0 = [&](int k) -> int { return pos_first + k * pos_step; };
    auto tile_interior = [&](int pos0) -> bool { return pos0 >= 0 && pos0 + (FR_ROWS - 1) * P + pitch <= len32; };
    // start the TMA copy of tile k into ring slot k % FR_STAGES (interior tiles only); the bookkeeping is
    // warp-uniform, only the two asynchronous instructions are issued by one lane
    // a tile that lies completely in the history is copied the same way from hist2 (same overlapping-row map) and
    // un-mixed in shared memory; only a tile that straddles the start or the end of the push is filled by hand
    const int hist32 = a.has_hist_map ? (int)hist_len : 0;
    auto tile_history = [&](int pos0) -> bool { return hist32 > 0 && pos0 >= -hist32 && pos0 + (FR_ROWS - 1) * P + pitch <= 0; };
    auto issue = [&](int k) {
        const int pos0 = tile_pos0(k);
        const bool live = k < n_tiles;
        const bool from_in = live && tile_interior(pos0), from_hist = live && !from_in && tile_history(pos0);
        const uint32_t bar = bar0 + (k % FR_STAGES) * 8;
        if ((from_in || from_hist) && lane == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tile_bytes) : "memory");
            asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
                             tiles_s + (k % FR_STAGES) * tile_stride),
                         "l"(from_in ? &tmap : &tmap_h), "r"(bar), "r"(from_in ? pos0 : pos0 + hist32), "r"(0), "r"(SHARED_IN && from_in ? 0 : s)
                         : "memory");
        }
    };
#pragma unroll
    for (int q = 0; q < FR_STAGES - 1; ++q) issue(q);

    if (a.kept_rows > 0 && tile0 == 0) {
        // the history rows of u kept from the previous push (its buffer) move in front of this push's rows, while the
        // first tile is on its way
        const float4* __restrict__ src4 = reinterpret_cast<const float4*>(reinterpret_cast<const float2*>(a.kept_src) + (long long)s * a.kept_stride);
        float4* __restrict__ dst4 = u - (long long)a.kept_rows * RK / 2;
        for (int e = lane; e < a.kept_rows * RK / 2; e += 32) dst4[e] = __ldg(src4 + e);
    }

    uint32_t phase = 0;  // bit q: parity of ring slot q's next completion
    pc rowph(1.f, 0.f);
    for (int k = 0; k < n_tiles; ++k) {
        const int slot = k % FR_STAGES;
        const int v0 = (tile0 + k) * FR_ROWS;  // first row (of this push's u rows) of the tile
        const int pos0 = tile_pos0(k);
        const bool history = tile_history(pos0);
        const bool interior = tile_interior(pos0) || history;  // arrives by TMA
        const uint32_t tile_s = tiles_s + slot * tile_stride;
        // the slot of tile k + FR_STAGES - 1 was released at the end of the previous iteration
        issue(k + FR_STAGES - 1);
        // row phasor: exact at the warp's first tile and every 16th one, rotated in between
        if (HAS_NCO) {
            if ((k & 15) == 0) {
                long long kk = ((long long)idx0 + pos0 + (long long)row * P) % (long long)denom;
                if (kk < 0) kk += denom;
                const cx<float> c = nco_phasor<float>(mulmod_u32(numer_abs, (uint32_t)kk, denom), denom, sign, start);
                rowph = pc(c.x, c.y);
            } else {
                rowph = pcmul(rowph, rot_tile);
            }
        }
        if (interior) {
            asm volatile(
                "{\n"
                ".reg .pred p;\n"
                "FW_%=:\n"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                "@p bra FD_%=;\n"
                "bra FW_%=;\n"
                "FD_%=:\n"
                "}\n" ::"r"(bar0 + slot * 8),
                "r"((phase >> slot) & 1)
                : "memory");
            phase ^= 1u << slot;
            if (HAS_NCO && history) {
                // history samples are already mixed: give them the conjugate of the phasors applied below
                float2* dst = reinterpret_cast<float2*>(tiles + slot * tile_stride);
                for (int r = 0; r < FR_ROWS; ++r) {
                    const pc rp(__shfl_sync(0xffffffffu, rowph.x, 2 * r), __shfl_sync(0xffffffffu, rowph.y, 2 * r));
                    for (int p = lane; p < P; p += 32) {
                        const float2 c = colph[p], q = dst[r * pitch + p];
                        const pc y = pcmulc(pc(q.x, q.y), pcmul(rp, pc(c.x, c.y)));
                        dst[r * pitch + p] = make_float2(y.x, y.y);
                    }
                }
                __syncwarp();
            }
        } else {
            // edge tile (reaches before the pushed samples or past them): the warp fills its slot itself,
            // coalesced.  History samples are already mixed: they get the conjugate of the phasors that the
            // loop below and the row's results apply.
            float2* dst = reinterpret_cast<float2*>(tiles + slot * tile_stride);
            constexpr int UNR = 13;  // loads in flight per lane: a 16 x 50 tile in two round trips
            for (int e0 = lane; e0 < FR_ROWS * P; e0 += 32 * UNR) {
                float2 q[UNR];
#pragma unroll
                for (int j = 0; j < UNR; ++j) {
                    const int e = e0 + 32 * j;
                    const long long pos = pos0 + e;
                    q[j] = make_float2(0.f, 0.f);
                    if (e < FR_ROWS * P) {
                        if (pos >= 0) {
                            if (pos < len) q[j] = __ldg(in + pos);
                        } else if (pos >= -hist_len) {
                            q[j] = __ldg(hist_end + pos);
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < UNR; ++j) {
                    const int e = e0 + 32 * j;
                    const int er = e < FR_ROWS * P ? e : 0;
                    const int rr_ = er / P, p = er - rr_ * P;
                    const int de = rr_ * pitch + p;  // position in the (possibly padded) tile
                    if (HAS_NCO) {
                        const float rx = __shfl_sync(0xffffffffu, rowph.x, 2 * rr_), ry = __shfl_sync(0xffffffffu, rowph.y, 2 * rr_);
                        if (pos0 + e < 0) {
                            const float2 c = colph[p];
                            const pc f = pcmul(pc(rx, ry), pc(c.x, c.y));
                            const pc y = pcmulc(pc(q[j].x, q[j].y), f);
                            q[j] = make_float2(y.x, y.y);
                        }
                    }
                    if (e < FR_ROWS * P) dst[de] = q[j];
                }
            }
            __syncwarp();
        }
        pc acc[RK];
#pragma unroll
        for (int c = 0; c < RK; ++c) acc[c] = pc(0.f, 0.f);
        const uint32_t row_s = tile_s + row * (pitch * 8);
        const long long prow = pos0 + (long long)row * P;  // push offset of this lane's row
        const bool row_ok = v0 + row < a.n_rows;
        // history samples leave either straight from the registers (8/16-byte pieces per lane: fine when few tiles do it)
        // or, when most tiles of the launch do, through the tile with coalesced stores
        const bool staged = a.hist_staged != 0;
        auto run_row = [&](auto write_hist) {
#pragma unroll 4
            for (int it = 0; it < cnt; ++it) {
                int st = st0 + rot + it;
                if (st >= st1) st -= cnt;
                pc x0, x1;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x0.x), "=f"(x0.y), "=f"(x1.x), "=f"(x1.y) : "r"(row_s + st * 16));
                if (HAS_NCO) {
                    pc c0, c1;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(c0.x), "=f"(c0.y), "=f"(c1.x), "=f"(c1.y) : "r"(col_s + st * 16));
                    x0 = pcmul(x0, c0);
                    x1 = pcmul(x1, c1);
                }
                if (decltype(write_hist)::value) {
                    // the Filter's next history = the fully mixed samples
                    const pc y0 = HAS_NCO ? pcmul(x0, rowph) : x0, y1 = HAS_NCO ? pcmul(x1, rowph) : x1;
                    if (staged) {
                        // parked in the tile (each lane overwrites what it has just read), written out row by row after the loop
                        if (HAS_NCO)
                            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(row_s + st * 16), "f"(y0.x), "f"(y0.y), "f"(y1.x), "f"(y1.y)
                                         : "memory");
                    } else {
                        const long long j = prow + 2 * st - a.hist_from;
                        if (row_ok && j >= -1 && j < hist_cap) {  // (a last row may reach past the pushed samples)
                            if (j >= 0) hist_o[j] = make_float2(y0.x, y0.y);
                            if (j + 1 < hist_cap) hist_o[j + 1] = make_float2(y1.x, y1.y);
                        }
                    }
                }
                float cf[2 * RK];
#pragma unroll
                for (int q = 0; q < (2 * RK) / 4; ++q)
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                                 : "=f"(cf[4 * q]), "=f"(cf[4 * q + 1]), "=f"(cf[4 * q + 2]), "=f"(cf[4 * q + 3])
                                 : "r"(coef_s + st * CP + q * 16));
#pragma unroll
                for (int c = 0; c < RK; ++c) {
                    acc[c] = pfma_s(x0, cf[c], acc[c]);
                    acc[c] = pfma_s(x1, cf[RK + c], acc[c]);
                }
            }
            if (odd_steps) {
                // the last column pair: one sample per lane
                const int p = 2 * full + hh;
                pc x0 = lds_front(row_s + p * 8);
                if (HAS_NCO) x0 = pcmul(x0, lds_front(col_s + p * 8));
                if (decltype(write_hist)::value) {
                    const pc y0 = HAS_NCO ? pcmul(x0, rowph) : x0;
                    if (staged) {
                        if (HAS_NCO) asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(row_s + p * 8), "f"(y0.x), "f"(y0.y) : "memory");
                    } else {
                        const long long j = prow + p - a.hist_from;
                        if (row_ok && j >= 0 && j < hist_cap) hist_o[j] = make_float2(y0.x, y0.y);
                    }
                }
                float cf[RK];
                static_assert(RK % 2 == 0, "coefficient rows are read in pairs");
#pragma unroll
                for (int q = 0; q < RK / 2; ++q)
                    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(cf[2 * q]), "=f"(cf[2 * q + 1]) : "r"(coef_s + (p >> 1) * CP + (p & 1) * (RK * 4) + q * 8));
#pragma unroll
                for (int c = 0; c < RK; ++c) acc[c] = pfma_s(x0, cf[c], acc[c]);
            }
        };
        const bool to_hist = hist_o != nullptr && pos0 + (long long)FR_ROWS * P > a.hist_from;
        if (to_hist) run_row(std::true_type{});
        else run_row(std::false_type{});
        if (to_hist && staged) {
            // rows are consecutive in the stream: coalesced 8-byte stores, a row per pass
            __syncwarp();
            const float2* src = reinterpret_cast<const float2*>(tiles + slot * tile_stride);
            const int rows_ok = min(FR_ROWS, a.n_rows - v0);
            for (int r = 0; r < rows_ok; ++r) {
                const long long j0 = (long long)pos0 + (long long)r * P - a.hist_from;
                for (int p = lane; p < P; p += 32)
                    if (j0 + p >= 0 && j0 + p < hist_cap) hist_o[j0 + p] = src[r * pitch + p];
            }
        }
        // every lane is done with the slot: it may be refilled (generic-proxy accesses ordered before the copy)
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        // the two column halves of a row meet; lane hh = 0 stores results [0, RK_SPLIT), lane hh = 1 the others
#pragma unroll
        for (int c = 0; c < RK; ++c)
            acc[c] = acc[c] + pc(__shfl_xor_sync(0xffffffffu, acc[c].x, 1), __shfl_xor_sync(0xffffffffu, acc[c].y, 1));
        const int v = v0 + row;
        if (v < a.n_rows) {
            float4* dst = u + ((long long)v * RK) / 2;
            if (hh == 0) {
#pragma unroll
                for (int c = 0; c < RK_SPLIT; c += 2) {
                    pc y0 = acc[c], y1 = acc[c + 1];
                    if (HAS_NCO) {
                        y0 = pcmul(y0, rowph);
                        y1 = pcmul(y1, rowph);
                    }
                    dst[c / 2] = make_float4(y0.x, y0.y, y1.x, y1.y);
                }
            } else {
#pragma unroll
                for (int c = RK_SPLIT; c < RK; c += 2) {
                    pc y0 = acc[c], y1 = acc[c + 1];
                    if (HAS_NCO) {
                        y0 = pcmul(y0, rowph);
                        y1 = pcmul(y1, rowph);
                    }
                    dst[c / 2] = make_float4(y0.x, y0.y, y1.x, y1.y);
                }
            }
        }
    }
}

using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                              const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn front_encode_fn() {
    static EncodeFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeFn>(p);
    });
    return fn;
}

}  // namespace

bool front_supported(int rank_pad, long long P) {
    // even P (TMA rows are 16-byte multiples; the tile pitch is padded to an odd number of 16-byte units); one TMA
    // box per tile
    return (rank_pad == 10 || rank_pad == 16) && P >= 2 && P <= 254 && (P % 2) == 0 && front_encode_fn() != nullptr;
}

cudaError_t launch_front(int rank_pad, int n_streams, const FrontArgs& a0, bool shared, cudaStream_t st) {
    EncodeFn enc = front_encode_fn();
    if (!enc || (rank_pad != 10 && rank_pad != 16)) return cudaErrorNotSupported;
    FrontArgs a = a0;
    const int tiles = (a.n_rows + FR_ROWS - 1) / FR_ROWS;
    // long-lived warps amortise the per-CTA tables: as few CTAs per stream as keep ~4 CTAs per SM in the
    // grid, the tiles spread evenly over their warps
    int ctas = (tiles + FR_WARPS * 64 - 1) / (FR_WARPS * 64);
    while ((long long)n_streams * ctas < 592 && ctas * FR_WARPS < tiles) ++ctas;
    a.tiles_per_warp = (tiles + ctas * FR_WARPS - 1) / (ctas * FR_WARPS);
    // the stream as overlapping rows of P samples: element (c0, i, s) = in[s*in_stride + c0 + i*P].  shared: one row
    // that every stream reads, mapped once (a zero stride cannot be encoded)
    if (shared != (n_streams > 1 && a.in_stride == 0)) return cudaErrorInvalidValue;
    CUtensorMap tm;
    const cuuint64_t dims[3] = {(cuuint64_t)a.len, (cuuint64_t)FR_ROWS, (cuuint64_t)(shared ? 1 : n_streams)};
    const cuuint64_t sstride = n_streams > 1 && !shared ? (cuuint64_t)a.in_stride * 8 : (((cuuint64_t)a.len * 8 + 15) / 16) * 16;
    const cuuint64_t strides[2] = {(cuuint64_t)a.P * 8, sstride};
    const int pitch = a.P + ((a.P & 3) == 0 ? 2 : 0);
    const cuuint32_t box[3] = {(cuuint32_t)pitch, (cuuint32_t)FR_ROWS, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<void*>(a.in), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    // the history as the same kind of map: element (c0, i, s) = hist2[s*2n + c0 + i*P]
    CUtensorMap tmh = tm;
    a.has_hist_map = 0;
    if (a.hist2 && a.n > 0 && ((uintptr_t)a.hist2 % 16) == 0 && 2 * a.n >= (long long)FR_ROWS * a.P + pitch) {
        const cuuint64_t hdims[3] = {(cuuint64_t)(2 * a.n), (cuuint64_t)FR_ROWS, (cuuint64_t)n_streams};
        const cuuint64_t hstrides[2] = {(cuuint64_t)a.P * 8, (cuuint64_t)(2 * a.n) * 8};
        if (enc(&tmh, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<void*>(a.hist2), hdims, hstrides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
            a.has_hist_map = 1;
    }
    const int tile_stride = (FR_ROWS * pitch * 8 + 127) / 128 * 128;
    const size_t smem = (size_t)FR_WARPS * FR_STAGES * tile_stride + (size_t)(a.P / 2 + 1) * front_coef_pitch(rank_pad) + (size_t)a.P * 8 + FR_WARPS * FR_STAGES * 8 + 16;
    const dim3 grid((unsigned)((tiles + FR_WARPS * a.tiles_per_warp - 1) / (FR_WARPS * a.tiles_per_warp)), (unsigned)n_streams);
    cudaError_t e = cudaSuccess;
    auto go = [&](auto kern) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) kern<<<grid, FR_WARPS * 32, smem, st>>>(tm, tmh, a);
    };
    if (rank_pad == 10) {
        if (shared) {
            if (a.nco) go(k_front<10, true, true>);
            else go(k_front<10, false, true>);
        } else {
            if (a.nco) go(k_front<10, true, false>);
            else go(k_front<10, false, false>);
        }
    } else {
        if (shared) {
            if (a.nco) go(k_front<16, true, true>);
            else go(k_front<16, false, true>);
        } else {
            if (a.nco) go(k_front<16, true, false>);
            else go(k_front<16, false, false>);
        }
    }
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

}  // namespace rr
