// k_fused: FreqShifter -> Filter -> Downsampler (integer decimation P, complex f32) in ONE persistent kernel.
//
// Same algebra as k_front + k_poly2 (rr_front.cu, rr_poly2.cu: the fused filter's P x (Lmax+1) matrix is
// sum_c a_c b_c^T to below f32 rounding), but the intermediate u never travels through HBM:
//
//   front-end warps (F):  u_c[i] = rowph(i) * sum_p a_c[p] * colph(p) * x[iP + p]   -> rows of a shared-memory tile
//   transform warps (T):  y = sum_c (b_c * u_c)  by 512-point overlap-save transforms on that tile -> HBM
//
// so a step reads every input sample once (8 B) and writes every output once (8 B / P): the algorithmic bytes of
// SURVEY.md 8d.  One CTA per SM walks through whole streams; per stream the two roles meet at two tile stages
// guarded by full/empty mbarriers, a block of V = 511 - Lmax new rows each.
//
// F warp: one lane per row of P samples (32 rows = one tile), so the RK x P coefficients are warp-uniform and come
// from constant memory through the uniform datapath (LDCU -> FFMA2 with a uniform-register operand): no
// shared-memory traffic for them (k_front's coefficient reads took 20 of its 28 wavefronts per step and made it
// LSU bound).  Samples arrive by TMA, half a row per box (two boxes of `hp` columns per tile), into a per-warp
// ring of slots with its own mbarriers; a warp runs ahead over stream boundaries.
//
// T warps: k_poly2's SINGLE path (two columns per warp end to end, one exchange, products summed through the
// stage, spectra parked, inverse transforms in groups), fed from the stage instead of a TMA tile.  The Lmax rows a
// block shares with its predecessor are carried in each warp's own 16-byte strip (a small keep buffer); the first
// block of a stream takes them from the rows the previous push kept in HBM.
//
// Reference semantics: transform.rs:333-348 (NCO), filters.rs:240-253 (overlap-save Filter),
// resampling.rs:103-121 (decimating FIR).  sm_100a only.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "rr_kernels.h"
#include "rr_poly.cuh"
#include "rr_pk.cuh"

namespace rr {

namespace {

constexpr int FK = 512;          // points per transform
constexpr int FRK = 10;          // columns of u (rank of the factorisation, padded)
constexpr int T_WARPS = FRK / 2;  // transform warps: two columns each
constexpr int T_THREADS = 32 * T_WARPS;
constexpr int F_ROWS = 32;       // rows per front-end tile: one lane per row
constexpr int PITCH = FRK * 8;   // bytes per stage row
constexpr int STAGE_ROWS = 528;  // 512 + spare rows of the exchange layout (element (t, k1) at row 33 t + k1)
constexpr int STAGE_BYTES = STAGE_ROWS * PITCH;
constexpr int TW_UNITS = 17;
constexpr int TW_BYTES = 16 * TW_UNITS * 16;
constexpr int YS_STRIDE = FK + 1;

// coefficient tables in constant memory: kFusedSlots tables of up to kFusedSlotFloats floats ([P/2][2][FRK])
constexpr int kFusedSlots = 6;
constexpr int kFusedSlotFloats = 2560;  // P <= 256
__constant__ float4 c_fcoef[kFusedSlots * kFusedSlotFloats / 4];

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mb_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mb_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "FWAIT_%=:\n"
        "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%0], %1;\n"
        "@p bra FDONE_%=;\n"
        "bra FWAIT_%=;\n"
        "FDONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// the same for waits that are expected to be long (a transform warp waiting for its block to be filled: ~60 % of its
// time): the suspend-time hint lets the hardware park the warp instead of re-issuing the test (the retries of the plain
// form were 7 % of all issued instructions and compete with the front-end warps of the same scheduler)
__device__ __forceinline__ void mb_wait_long(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LWAIT_%=:\n"
        "mbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra LDONE_%=;\n"
        "bra LWAIT_%=;\n"
        "LDONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity), "r"(20000u)
        : "memory");
}
__device__ __forceinline__ pc f_lds(uint32_t addr) {
    pc r;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(addr));
    return r;
}
__device__ __forceinline__ void f_lds2(uint32_t addr, pc& a, pc& b) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(b.x), "=f"(b.y) : "r"(addr));
}
__device__ __forceinline__ void f_sts(uint32_t addr, pc a) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a.x), "f"(a.y) : "memory");
}
__device__ __forceinline__ void f_sts2(uint32_t addr, pc a, pc b) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y) : "memory");
}
__device__ __forceinline__ void f_ldg2(const float4* p, pc& a, pc& b) {
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(b.x), "=f"(b.y) : "l"(p));
}

// exp(j * sign * 2*pi * (numer*d mod denom) / denom), the phase advance over d samples: rr_poly.cuh's nco_rotation (same
// integer phase, same double-precision evaluation) without its 64-bit divisions; inv_m = 1 / denom
__device__ __forceinline__ pc f_rotation(uint32_t d, uint32_t numer_abs, uint32_t denom, double inv_m, int sign) {
    const uint32_t r = mulmod_fast(numer_abs, d % denom, denom, inv_m);
    double s, c;
    sincospi(2.0 * (double)r / (double)denom, &s, &c);
    return pc((float)c, (float)(sign < 0 ? -s : s));
}

// pass 1 of the 512-point transform of this thread's 32 inputs (rows t + 16*i1), as in rr_poly2.cu
__device__ __forceinline__ void f_pass1_store(pc (&v)[32], uint32_t tw_row, uint32_t xch_wr) {
    pdft_regs<32, +1>(v);
    pc w[3][2];
    f_lds2(tw_row, w[0][0], w[0][1]);
    f_lds2(tw_row + 16, w[1][0], w[1][1]);
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        if (m + 2 < 16) f_lds2(tw_row + (m + 2) * 16, w[(m + 2) % 3][0], w[(m + 2) % 3][1]);
        f_sts(xch_wr + (2 * m) * PITCH, pcmul(v[2 * m], w[m % 3][0]));
        f_sts(xch_wr + (2 * m + 1) * PITCH, pcmul(v[2 * m + 1], w[m % 3][1]));
    }
}

// RR_FUSED_PROF: per-phase cycle counters of front-end warp 0 / transform warp 0 of every CTA (development builds only)
#ifdef RR_FUSED_PROF
#define PROF(...) __VA_ARGS__
__device__ long long g_fused_prof[256 * 16];
#else
#define PROF(...)
#endif

struct FusedGeom {
    int steps, S0, hp, slot_bytes, slot_stride;  // column pairs per row, pairs in half 0, box columns, ring slot size
};
__host__ __device__ inline FusedGeom fused_geom(int P) {
    FusedGeom g;
    g.steps = P / 2;
    g.S0 = (g.steps + 1) / 2;
    g.hp = 2 * g.S0 + ((g.S0 & 1) ? 0 : 2);  // an odd number of 16-byte units per slot row: conflict-free 16-byte row loads
    if (g.hp > P) g.hp = P;
    g.slot_bytes = F_ROWS * g.hp * 8;
    g.slot_stride = (g.slot_bytes + 127) / 128 * 128;
    return g;
}

// steps [S_LO, S_HI) of a row, fully unrolled: the coefficient addresses are kernel parameter + immediate, so the
// loads are LDCU (uniform datapath) and the compiler pipelines them and the shared-memory loads freely
template <int S_LO, int S_HI, bool HAS_NCO>
__device__ __forceinline__ void f_steps(pc (&acc)[FRK], const float4* __restrict__ xrow, const float4* __restrict__ crow, const float4* cf_base) {
#pragma unroll
    for (int st = S_LO; st < S_HI; ++st) {
        const float4 xv = xrow[st];
        pc x0(xv.x, xv.y), x1(xv.z, xv.w);
        if (HAS_NCO) {
            const float4 cv = crow[st];
            x0 = pcmul(x0, pc(cv.x, cv.y));
            x1 = pcmul(x1, pc(cv.z, cv.w));
        }
        const float4* cf = cf_base + st * 5;
        const float4 a0 = cf[0], a1 = cf[1], a2 = cf[2], a3 = cf[3], a4 = cf[4];
        const float k0[FRK] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y};
        const float k1[FRK] = {a2.z, a2.w, a3.x, a3.y, a3.z, a3.w, a4.x, a4.y, a4.z, a4.w};
#pragma unroll
        for (int c = 0; c < FRK; ++c) {
            acc[c] = pfma_s(x0, k0[c], acc[c]);
            acc[c] = pfma_s(x1, k1[c], acc[c]);
        }
    }
}

}  // namespace

// FW front-end warps, ring depth D per warp, NB parked spectra per inverse round; PT: decimation factor known at
// compile time (the front end's step loop is unrolled completely) or 0 (any even P); SHARED_IN: every stream reads
// the same input row (the tensor map holds that one row, the copies address stream 0)
template <int FW, int D, int NB, bool HAS_NCO, int PT, bool SHARED_IN>
__global__ void __launch_bounds__(T_THREADS + 32 * FW, 1)
k_fused(const __grid_constant__ CUtensorMap tmap, const FusedArgs a, const int n_streams) {
    extern __shared__ __align__(128) unsigned char smem[];
    // the warp index through a warp broadcast: the compiler then knows that role dispatch and everything derived from
    // it is warp-uniform (uniform registers, LDCU for the coefficient table)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int P = PT > 0 ? PT : a.P;
    const FusedGeom geo = fused_geom(P);
    const int Lmax = a.Lmax, V = a.V, n_out = a.n_out;
    const int B = (n_out + V - 1) / V;                       // blocks per stream
    const int n_tiles = (B * V + F_ROWS - 1) / F_ROWS;       // tiles per stream (rows >= n_out are written as zeros)

    // ---- shared-memory map ------------------------------------------------------------------------------
    const int keep_bytes = ((Lmax * PITCH) + 127) / 128 * 128;
    unsigned char* const p_stage = smem;
    unsigned char* const p_tw = p_stage + 2 * STAGE_BYTES;
    unsigned char* const p_keep = p_tw + TW_BYTES;
    unsigned char* const p_ys = p_keep + keep_bytes;
    unsigned char* const p_ring = p_ys + (((size_t)NB * YS_STRIDE * 8 + 127) / 128 * 128);
    unsigned char* const p_colph = p_ring + (size_t)FW * D * geo.slot_stride;
    unsigned char* const p_bar = p_colph + (((size_t)FW * P * 8 + 127) / 128 * 128);
    const uint32_t bar_full = s_u32(p_bar), bar_empty = bar_full + 16, bar_ring = bar_full + 32;
    const uint32_t left_cnt = bar_ring + FW * D * 8;  // per stage: transform warps that have left it (two 32-bit counters)

    // ---- one-time set-up: zero the stages (stale rows must be finite), twiddles, barriers ----------------------
    for (int e = threadIdx.x; e < 2 * STAGE_BYTES / 16; e += blockDim.x) reinterpret_cast<float4*>(p_stage)[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    {
        const float2* __restrict__ twK = reinterpret_cast<const float2*>(a.twK);
        for (int e = threadIdx.x; e < FK; e += blockDim.x) {
            const int tr = e >> 5, k1 = e & 31;
            const float2 w = twK[(tr * k1) & (FK - 1)];
            const int off = (tr * TW_UNITS + (k1 >> 1)) * 16 + (k1 & 1) * 8;
            *reinterpret_cast<float2*>(p_tw + off) = w;
        }
    }
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
        mb_init(bar_full, FW);
        mb_init(bar_full + 8, FW);
        mb_init(bar_empty, T_WARPS);
        mb_init(bar_empty + 8, T_WARPS);
        for (int q = 0; q < FW * D; ++q) mb_init(bar_ring + q * 8, 1);
        asm volatile("st.shared.v2.u32 [%0], {%1, %1};" ::"r"(left_cnt), "r"(0u) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int n_my = (n_streams - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;  // streams of this CTA
    if (n_my <= 0) return;

    if (warp >= T_WARPS) {
        // =====================================================================================================
        // front-end warps.  All bookkeeping is 32-bit and incremental (no divisions in the tile loop): the tile loop's
        // overhead competes with 25 steps of ~65 cycles.
        // =====================================================================================================
        const int fw = warp - T_WARPS;
        const uint32_t ring_s = s_u32(p_ring) + fw * (D * geo.slot_stride);
        const uint32_t rbar = bar_ring + fw * (D * 8);
        float2* const colph = reinterpret_cast<float2*>(p_colph) + fw * P;
        const int steps = geo.steps, S0 = geo.S0, hp = geo.hp;
        const int half1_col0 = P - hp;  // half 1's box covers columns [P - hp, P): it never reaches past the row
        const int J0 = (int)a.J0;
        const int hist_len = (int)(2 * a.n);
        const int hist_from = (int)a.hist_from;
        // Tile j of the CTA's stream number so belongs to warp (j + so * n_live) mod FW, n_live = the tiles with a valid row:
        // the live tiles of consecutive streams go round the warps without a gap.  (A one-chunk push has three live tiles
        // per stream: without the rotation three of the warps would do all the work.)
        const int n_live = (n_out + F_ROWS - 1) / F_ROWS;
        const int rot_step = n_live % FW;
        auto tiles_from = [&](int j0) { return j0 < n_tiles ? (n_tiles - j0 + FW - 1) / FW : 0; };  // tiles j0, j0 + FW, ... below n_tiles
        const int BV = B * V;
        const int tile_step = FW * F_ROWS;  // rows between consecutive tiles of this warp

        // ---- issue side: (stream ordinal, tile, half) of the next copy, its ring slot ------------------------------
        int i_so = 0, i_k = 0, i_half = 0, i_slot = 0;
        int i_j0 = fw, i_rot = 0, i_tw = tiles_from(fw);  // first tile, rotation and tile count of this warp in stream i_so
        auto issue_next = [&]() {
            // advance to the next item that has a copy (tiles with no valid row have none) and start it
            while (i_so < n_my) {
                if (i_k >= i_tw) {  // on to the next stream
                    ++i_so;
                    i_k = 0;
                    i_rot += rot_step;
                    if (i_rot >= FW) i_rot -= FW;
                    i_j0 = fw - i_rot + (fw < i_rot ? FW : 0);
                    i_tw = tiles_from(i_j0);
                    continue;
                }
                const int j = i_j0 + i_k * FW, half = i_half, so = i_so;
                i_half ^= 1;
                if (i_half == 0) ++i_k;
                const int rows_ok = min(F_ROWS, n_out - j * F_ROWS);
                if (rows_ok <= 0) continue;
                const int pos0 = j * (F_ROWS * P) - J0;
                const int coff = half ? half1_col0 : 0;
                // coordinates (c, i): address = c + i*P.  Rows that must not be read get a row coordinate outside
                // [0, F_ROWS) and are zero-filled: the rows behind the last valid one (tail), and row 0 of a tile
                // that starts before the pushed samples (head; patched by hand when the tile is consumed)
                const int sh = pos0 < 0 ? -1 : F_ROWS - rows_ok;
                if (lane == 0) {
                    mb_expect_tx(rbar + i_slot * 8, (uint32_t)geo.slot_bytes);
                    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
                                     ring_s + i_slot * geo.slot_stride),
                                 "l"(&tmap), "r"(rbar + i_slot * 8), "r"(pos0 + coff - sh * P), "r"(sh), "r"(SHARED_IN ? 0 : (int)blockIdx.x + so * (int)gridDim.x)
                                 : "memory");
                }
                i_slot = (i_slot + 1 == D) ? 0 : i_slot + 1;
                return;
            }
        };
#pragma unroll 1
        for (int q = 0; q < D; ++q) issue_next();

        PROF(long long pr[8] = {0, 0, 0, 0, 0, 0, 0, 0}; const long long pr_t0 = clock64();)
        int c_slot = 0;
        uint32_t c_phase = 0;  // parity of the consume slot's next completion (flips when the ring wraps)
        int gb_acq = -1;       // highest global block whose stage this warp has acquired
        int gb_arr = -1;       // highest global block this warp has arrived on (full)
        // arrive on `full` for every block up to gb_done: a block is only arrived on once its stage has been acquired
        // (i.e. the block two before is consumed), so that arrivals never pile up within one barrier phase
        auto arrive_upto = [&](int gb_done) {
            for (int g2 = gb_arr + 1; g2 <= gb_done; ++g2) {
                while (gb_acq < g2) {
                    ++gb_acq;
                    mb_wait(bar_empty + (uint32_t)(gb_acq & 1) * 8, (uint32_t)(((gb_acq >> 1) & 1) ^ 1));
                }
                __syncwarp();
                if (lane == 0) mb_arrive(bar_full + (uint32_t)(g2 & 1) * 8);
            }
            if (gb_done > gb_arr) gb_arr = gb_done;
        };

        int rot = 0;  // so * n_live mod FW
#pragma unroll 1
        for (int so = 0; so < n_my; ++so) {
            PROF(const long long pst0 = clock64();)
            const int s = (int)blockIdx.x + so * (int)gridDim.x;
            const int gb0 = so * B;  // global index of this stream's block 0
            const int j0 = fw - rot + (fw < rot ? FW : 0);  // this warp's first tile of the stream
            const int tiles_w = tiles_from(j0);
            rot += rot_step;
            if (rot >= FW) rot -= FW;
            // ---- per-stream NCO constants -------------------------------------------------------------
            uint32_t denom = 1, numer_abs = 0, idx0 = 0;
            int sign = 0;
            float start = 0.f;
            pc rot_tile(1.f, 0.f);
            double inv_denom = 1.0;
            if (HAS_NCO && j0 < n_live) {  // (a warp without a live tile in this stream needs none of it)
                const NcoStream ns = a.nco[s];
                denom = ns.denom;
                numer_abs = ns.numer_abs;
                sign = ns.sign;
                idx0 = ns.idx;
                start = (float)ns.start_phase;
                inv_denom = 1.0 / (double)denom;
                rot_tile = f_rotation((uint32_t)(tile_step * P), numer_abs, denom, inv_denom, sign);
                __syncwarp();  // the previous stream's column phasors are no longer read
                for (int p = lane; p < P; p += 32) {
                    const pc c = f_rotation((uint32_t)p, numer_abs, denom, inv_denom, sign);
                    colph[p] = make_float2(c.x, c.y);
                }
                __syncwarp();
            }
            const float2* __restrict__ in = reinterpret_cast<const float2*>(a.in) + (long long)s * a.in_stride;
            const float2* __restrict__ hist_end = reinterpret_cast<const float2*>(a.hist2) + ((long long)s + 1) * hist_len;
            float2* __restrict__ hist_o = a.hist_out ? reinterpret_cast<float2*>(a.hist_out) + (long long)s * a.hist_stride : nullptr;
            float4* __restrict__ keep_o = reinterpret_cast<float4*>(reinterpret_cast<float2*>(a.ukeep_out) + (long long)s * a.ukeep_out_stride);
            const float4* cf_base = c_fcoef + a.coef_off4;
            const float4* __restrict__ crow = reinterpret_cast<const float4*>(colph);

            PROF(pr[7] += clock64() - pst0;)
            // block and offset within the block of the tile's first row
            int blk = (j0 * F_ROWS) / V, off = (j0 * F_ROWS) - blk * V;
            pc rowph(1.f, 0.f);
#pragma unroll 1
            for (int k = 0; k < tiles_w; ++k) {
                const int r0 = (j0 + k * FW) * F_ROWS;  // first row of the tile
                const int row = r0 + lane;              // this lane's row
                const int pos0 = r0 * P - J0;
                pc acc[FRK];
#pragma unroll
                for (int c = 0; c < FRK; ++c) acc[c] = pc(0.f, 0.f);
                PROF(long long pc0 = clock64();)
                if (r0 < n_out) {
                    if (HAS_NCO) {
                        if ((k & 15) == 0) {
                            // table index (idx0 + offset of the row) mod denom, without a 64-bit division
                            const long long v = (long long)idx0 + pos0 + (long long)lane * P;
                            long long kk = v - (long long)floor((double)v * inv_denom) * (long long)denom;
                            if (kk < 0) kk += denom;
                            else if (kk >= (long long)denom) kk -= denom;
                            const cx<float> c = nco_phasor<float>(mulmod_fast(numer_abs, (uint32_t)kk, denom, inv_denom), denom, sign, start);
                            rowph = pc(c.x, c.y);
                        } else {
                            rowph = pcmul(rowph, rot_tile);
                        }
                    }
                    const int prow = pos0 + lane * P;  // push offset of this lane's row
                    const bool to_hist = hist_o != nullptr && pos0 + F_ROWS * P > hist_from;
#pragma unroll 1
                    for (int half = 0; half < 2; ++half) {
                        const uint32_t slot_s = ring_s + c_slot * geo.slot_stride;
                        PROF(long long pw0 = clock64(); pr[0] += pw0 - pc0;)
                        mb_wait(rbar + c_slot * 8, c_phase);
                        PROF(long long pw1 = clock64(); pr[1] += pw1 - pw0;)
                        const int col0 = half ? half1_col0 : 0;
                        if (pos0 < 0) {
                            // head tile: row 0 arrived as zeros; fill it from the history (already mixed: un-mix) and the push
                            float2* dst = reinterpret_cast<float2*>(smem + (slot_s - s_u32(smem)));
                            const float r0x = __shfl_sync(0xffffffffu, rowph.x, 0), r0y = __shfl_sync(0xffffffffu, rowph.y, 0);
                            for (int cc = lane; cc < hp; cc += 32) {
                                const int p = col0 + cc;
                                const int pos = pos0 + p;
                                float2 q = make_float2(0.f, 0.f);
                                if (pos >= 0) {
                                    if (pos < (int)a.len) q = __ldg(in + pos);
                                } else if (pos >= -hist_len) {
                                    q = __ldg(hist_end + pos);
                                    if (HAS_NCO) {
                                        const float2 cph = colph[p];
                                        const pc y = pcmulc(pc(q.x, q.y), pcmul(pc(r0x, r0y), pc(cph.x, cph.y)));
                                        q = make_float2(y.x, y.y);
                                    }
                                }
                                dst[cc] = q;
                            }
                            __syncwarp();
                        }
                        // plain (non-volatile) shared-memory loads: the compiler pipelines them and the constant-bank loads
                        // over the unrolled steps; the mbarrier wait above (memory clobber) keeps them behind the copy.
                        // slot column of sample column 2*st: 2*st - col0
                        const float4* __restrict__ xrow = reinterpret_cast<const float4*>(smem + (slot_s - s_u32(smem)) + lane * (hp * 8) - col0 * 8);
                        if (to_hist) {
                            // tiles inside the last 2n samples: the Filter's next history = the fully mixed samples
                            // (filters.rs:260 keeps the input chunk); a few tiles per stream, run-time loop
                            const int st_lo = half ? S0 : 0, st_hi = half ? steps : S0;
#pragma unroll 2
                            for (int st = st_lo; st < st_hi; ++st) {
                                const float4 xv = xrow[st];
                                pc x0(xv.x, xv.y), x1(xv.z, xv.w);
                                if (HAS_NCO) {
                                    const float4 cv = crow[st];
                                    x0 = pcmul(x0, pc(cv.x, cv.y));
                                    x1 = pcmul(x1, pc(cv.z, cv.w));
                                }
                                const pc y0 = HAS_NCO ? pcmul(x0, rowph) : x0, y1 = HAS_NCO ? pcmul(x1, rowph) : x1;
                                const int jh = prow + 2 * st - hist_from;
                                if (row < n_out && jh >= -1) {
                                    if (jh >= 0) hist_o[jh] = make_float2(y0.x, y0.y);
                                    hist_o[jh + 1] = make_float2(y1.x, y1.y);
                                }
                                const float4* cf = cf_base + st * 5;
                                const float4 a0 = cf[0], a1 = cf[1], a2 = cf[2], a3 = cf[3], a4 = cf[4];
                                const float k0[FRK] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y};
                                const float k1[FRK] = {a2.z, a2.w, a3.x, a3.y, a3.z, a3.w, a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                                for (int c = 0; c < FRK; ++c) {
                                    acc[c] = pfma_s(x0, k0[c], acc[c]);
                                    acc[c] = pfma_s(x1, k1[c], acc[c]);
                                }
                            }
                        } else if constexpr (PT > 0) {
                            constexpr int STEPS_C = PT / 2, S0_C = (STEPS_C + 1) / 2;
                            if (half == 0) f_steps<0, S0_C, HAS_NCO>(acc, xrow, crow, cf_base);
                            else f_steps<S0_C, STEPS_C, HAS_NCO>(acc, xrow, crow, cf_base);
                        } else {
                            const int st_lo = half ? S0 : 0, st_hi = half ? steps : S0;
#pragma unroll 4
                            for (int st = st_lo; st < st_hi; ++st) {
                                const float4 xv = xrow[st];
                                pc x0(xv.x, xv.y), x1(xv.z, xv.w);
                                if (HAS_NCO) {
                                    const float4 cv = crow[st];
                                    x0 = pcmul(x0, pc(cv.x, cv.y));
                                    x1 = pcmul(x1, pc(cv.z, cv.w));
                                }
                                const float4* cf = cf_base + st * 5;
                                const float4 a0 = cf[0], a1 = cf[1], a2 = cf[2], a3 = cf[3], a4 = cf[4];
                                const float k0[FRK] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y};
                                const float k1[FRK] = {a2.z, a2.w, a3.x, a3.y, a3.z, a3.w, a4.x, a4.y, a4.z, a4.w};
#pragma unroll
                                for (int c = 0; c < FRK; ++c) {
                                    acc[c] = pfma_s(x0, k0[c], acc[c]);
                                    acc[c] = pfma_s(x1, k1[c], acc[c]);
                                }
                            }
                        }
                        // every lane is done with the slot: refill it (generic-proxy reads ordered before the async copy)
                        PROF(long long ps1 = clock64(); pr[2] += ps1 - pw1;)
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        PROF(long long ps2 = clock64(); pr[3] += ps2 - ps1;)
                        if (++c_slot == D) {
                            c_slot = 0;
                            c_phase ^= 1u;
                        }
                        issue_next();
                        PROF(pc0 = clock64(); pr[4] += pc0 - ps2;)
                    }
                }
                // ---- the tile's rows go to the stage(s) of their block(s) -------------------------------------
                {
                    const int last_off = min(off + F_ROWS, BV - blk * V) - 1;  // offset (from block blk's first row) of the tile's last row below B*V
                    const int gb_hi = gb0 + blk + (last_off >= V ? 1 : 0);
                    PROF(long long pe0 = clock64(); pr[0] += pe0 - pc0;)
                    while (gb_acq < gb_hi) {
                        ++gb_acq;
                        // free when the transform warps have released the block two before (passes at once for the first two)
                        mb_wait(bar_empty + (uint32_t)(gb_acq & 1) * 8, (uint32_t)(((gb_acq >> 1) & 1) ^ 1));
                    }
                    PROF(pc0 = clock64(); pr[5] += pc0 - pe0;)
                }
                if (row < BV) {
                    int b = blk, o = off + lane;
                    if (o >= V) {
                        o -= V;
                        ++b;
                    }
                    const uint32_t dst = s_u32(p_stage) + (uint32_t)((gb0 + b) & 1) * STAGE_BYTES + (Lmax + o) * PITCH;
                    const bool live = row < n_out;
                    const bool keep = live && row >= n_out - Lmax;  // the last Lmax rows of the push are the next push's history rows
#pragma unroll
                    for (int c = 0; c < FRK; c += 2) {
                        pc y0 = acc[c], y1 = acc[c + 1];
                        if (HAS_NCO) {
                            y0 = pcmul(y0, rowph);
                            y1 = pcmul(y1, rowph);
                        }
                        if (!live) {
                            y0 = pc(0.f, 0.f);
                            y1 = pc(0.f, 0.f);
                        }
                        f_sts2(dst + c * 8, y0, y1);
                        if (keep) keep_o[((row - (n_out - Lmax)) * FRK + c) / 2] = make_float4(y0.x, y0.y, y1.x, y1.y);
                    }
                }
                __syncwarp();
                // next tile of this warp; the blocks it no longer has rows for are complete on this warp's part
                off += tile_step;
                while (off >= V) {
                    off -= V;
                    ++blk;
                }
                arrive_upto((k + 1 < tiles_w) ? gb0 + min(blk, B) - 1 : gb0 + B - 1);
                PROF(pr[6] += clock64() - pc0;)
            }
            if (tiles_w == 0) arrive_upto(gb0 + B - 1);  // a warp without tiles (fewer tiles than warps) still owes its arrivals
        }
        PROF(if (fw == 0 && lane == 0) {
            for (int q = 0; q < 7; ++q) g_fused_prof[blockIdx.x * 16 + q] = pr[q];
            g_fused_prof[blockIdx.x * 16 + 7] = pr[7];
            g_fused_prof[blockIdx.x * 16 + 8] = clock64() - pr_t0;
        })
        return;
    }

    // =========================================================================================================
    // transform warps
    // =========================================================================================================
    const int tid = threadIdx.x;  // 0 .. T_THREADS-1
    const int t = lane >> 1, gg = lane & 1;
    const int g = 2 * warp + gg;  // column of u
    auto sync_t = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(T_THREADS) : "memory"); };
    const uint32_t stage0 = s_u32(p_stage);
    const uint32_t tw_row = s_u32(p_tw) + t * (TW_UNITS * 16);
    const uint32_t tile_rd = t * PITCH + g * 8;
    const uint32_t xch_wr = 33 * t * PITCH + g * 8;
    const uint32_t xch_rd = t * PITCH + g * 8;
    const uint32_t keep_s = s_u32(p_keep) + warp * 16;
    float2* const ysave = reinterpret_cast<float2*>(p_ys);
    const float4* __restrict__ gtab = reinterpret_cast<const float4*>(a.gtab);
    const int hist_rows_per_lane = (Lmax + 31) / 32;  // <= 12 (Lmax <= 383)

    const int n_blocks_total = n_my * B;
    // The Lmax rows of u the previous push kept enter rows [0, Lmax) of the stage of a stream's first block by one bulk copy
    // that completes on the stage's `full` barrier (the block then arrives whole, and no transform warp holds history rows
    // in registers over the wait).  It is started the moment the stage falls free: by the transform warp that is last to
    // leave it, before that warp's arrival on `empty` (so no front-end warp can have passed it), two blocks ahead.
    auto copy_kept = [&](int so_k, int gb_k) {
        const uint32_t bytes = (uint32_t)(Lmax * PITCH), bar = bar_full + (uint32_t)(gb_k & 1) * 8;
        const float2* src = reinterpret_cast<const float2*>(a.ukeep_in) + (long long)((int)blockIdx.x + so_k * (int)gridDim.x) * a.ukeep_in_stride;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the stage's rows were last written by ordinary stores
        asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(stage0 + (uint32_t)(gb_k & 1) * STAGE_BYTES),
                     "l"(src), "r"(bytes), "r"(bar)
                     : "memory");
    };
    if (tid == 0) {
        copy_kept(0, 0);
        if (B == 1 && n_my > 1) copy_kept(1, 1);
    }
    int parked = 0;      // spectra waiting for their inverse transform
    int gb_first = 0;    // global block of parked job 0
    int so = 0, b = -1;  // stream ordinal and block of the current global block
    PROF(long long tp[6] = {0, 0, 0, 0, 0, 0}; long long tc = clock64();)

#pragma unroll 1
    for (int gb = 0; gb < n_blocks_total; ++gb) {
        if (++b == B) {
            b = 0;
            ++so;
        }
        const int s = (int)blockIdx.x + so * (int)gridDim.x;
        const uint32_t stg = stage0 + (uint32_t)(gb & 1) * STAGE_BYTES;

        PROF({ long long n_ = clock64(); tp[0] += n_ - tc; tc = n_; })
        mb_wait_long(bar_full + (uint32_t)(gb & 1) * 8, (uint32_t)((gb >> 1) & 1));
        PROF({ long long n_ = clock64(); tp[1] += n_ - tc; tc = n_; })
        // rows [0, Lmax) of this warp's strip: the stream's first block has them in the stage already (the rows the previous
        // push kept, copied in by the front-end warp of tile 0), later blocks take them from the keep buffer, where rows
        // [V, V + Lmax) of every block's strip go for its successor
#pragma unroll
        for (int q = 0; q < 12; ++q) {
            const int r = lane + 32 * q;
            if (q < hist_rows_per_lane && r < Lmax) {
                float4 nx;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(nx.x), "=f"(nx.y), "=f"(nx.z), "=f"(nx.w) : "r"(stg + (V + r) * PITCH + warp * 16));
                if (b != 0) {
                    float4 h;
                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(h.x), "=f"(h.y), "=f"(h.z), "=f"(h.w) : "r"(keep_s + r * PITCH));
                    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(stg + r * PITCH + warp * 16), "f"(h.x), "f"(h.y), "f"(h.z), "f"(h.w) : "memory");
                }
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(keep_s + r * PITCH), "f"(nx.x), "f"(nx.y), "f"(nx.z), "f"(nx.w) : "memory");
            }
        }
        if (b == 0 && n_out < Lmax) {
            // a push with fewer new rows than the filter reaches back: the rows kept for the NEXT push are the tail of
            // [this push's history rows | its new rows]; the history part moves over here (this warp's strip of it), the
            // new rows are written by the front-end warps
            float4* __restrict__ kout = reinterpret_cast<float4*>(reinterpret_cast<float2*>(a.ukeep_out) + (long long)s * a.ukeep_out_stride);
#pragma unroll 1
            for (int r = n_out + lane; r < Lmax; r += 32) {
                float4 h;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(h.x), "=f"(h.y), "=f"(h.z), "=f"(h.w) : "r"(stg + r * PITCH + warp * 16));
                kout[((long long)(r - n_out) * FRK) / 2 + warp] = h;
            }
        }
        // row 511 takes part in the transform but in no stored output (the l = -1 slot of the low-rate filter is empty for
        // Q == 1): it must not hold what the previous block's exchange left there -- stale values of spectrum magnitude
        // would add their rounding noise to every output
        if (lane == 0) asm volatile("st.shared.v4.f32 [%0], {%1, %1, %1, %1};" ::"r"(stg + (FK - 1) * PITCH + warp * 16), "f"(0.f) : "memory");
        __syncwarp();

        // ---- forward transforms of this warp's two columns, products with FFT(b_c) ----------------------------------
        pc acc[32];
        {
            pc v[32];
            const uint32_t src = stg + tile_rd;
#pragma unroll
            for (int m = 0; m < 32; ++m) v[m] = f_lds(src + m * (16 * PITCH));
            __syncwarp();  // the strip's rows are consumed by every lane before any lane overwrites them
            f_pass1_store(v, tw_row, stg + xch_wr);
        }
        {
            const float4* gp = gtab + tid;
            pc h[16];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) f_ldg2(gp + jj * T_THREADS, h[2 * jj], h[2 * jj + 1]);
            __syncwarp();
#pragma unroll
            for (int which = 0; which < 2; ++which) {
                pc x[16];
#pragma unroll
                for (int tr = 0; tr < 16; ++tr) x[tr] = f_lds(stg + xch_rd + (33 * tr + 16 * which) * PITCH);
                pdft_regs<16, +1>(x);
#pragma unroll
                for (int k = 0; k < 16; ++k) acc[which * 16 + k] = pcmul(x[k], h[k]);
                if (which == 0) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) f_ldg2(gp + (8 + jj) * T_THREADS, h[2 * jj], h[2 * jj + 1]);
                }
            }
        }
        PROF({ long long n_ = clock64(); tp[2] += n_ - tc; tc = n_; })
        // ---- sum the ten partial spectra through the stage, park the block's spectrum ------------------------------
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; ++j) f_sts(stg + xch_rd + (16 * j) * PITCH, acc[j]);
        sync_t();
        if (parked == 0) gb_first = gb;
        {
            float2* ys = ysave + parked * YS_STRIDE;
            for (int o = tid; o < FK; o += T_THREADS) {
                const uint32_t src = stg + o * PITCH;
                pc sum(0.f, 0.f);
#pragma unroll
                for (int w = 0; w < T_WARPS; ++w) {
                    pc u0, u1;
                    f_lds2(src + w * 16, u0, u1);
                    sum = sum + u0;
                    sum = sum + u1;
                }
                const int j = o >> 4, tt = o & 15;
                ys[tt + 16 * (j >> 4) + 32 * (j & 15)] = make_float2(sum.x, sum.y);
            }
        }
        ++parked;
        PROF({ long long n_ = clock64(); tp[3] += n_ - tc; tc = n_; })

        // ---- inverse transforms of the parked spectra (column g takes job g), through the stage this block still holds
        if (parked == NB || gb + 1 == n_blocks_total) {
            sync_t();  // all sums are parked, nobody reads the stage's rows any more
#pragma unroll 1
            for (int j0 = 0; j0 < parked; j0 += FRK) {
                if (j0 + 2 * warp >= parked) continue;
                const int job = j0 + g;
                const bool active = job < parked;
                pc v[32];
                const float2* ys = ysave + (active ? job : 0) * YS_STRIDE;
#pragma unroll
                for (int i1 = 0; i1 < 32; ++i1) {
                    const float2 q = ys[t + 16 * i1];
                    v[i1] = active ? pc(q.x, -q.y) : pc(0.f, 0.f);  // conj in, conj out = inverse transform
                }
                f_pass1_store(v, tw_row, stg + xch_wr);
                __syncwarp();
                const int gj = gb_first + (active ? job : 0);
                const int so_j = gj / B, b_j = gj - so_j * B;
                const int s_j = (int)blockIdx.x + so_j * (int)gridDim.x;
                float2* __restrict__ out = reinterpret_cast<float2*>(a.out) + (long long)s_j * a.out_stride;
                float2* __restrict__ out2 = a.out2 ? reinterpret_cast<float2*>(a.out2) + (long long)s_j * a.out2_stride : nullptr;
#pragma unroll
                for (int which = 0; which < 2; ++which) {
                    pc x[16];
#pragma unroll
                    for (int tr = 0; tr < 16; ++tr) x[tr] = f_lds(stg + xch_rd + (33 * tr + 16 * which) * PITCH);
                    pdft_regs<16, +1>(x);
                    if (active) {
#pragma unroll
                        for (int k2 = 0; k2 < 16; ++k2) {
                            const int i = t + 16 * which + 32 * k2;
                            if (i >= Lmax && i < Lmax + V) {
                                const long long o = (long long)b_j * V + (i - Lmax);  // output index within the push
                                if (o < n_out) {
                                    float2* dst = (out2 != nullptr && o >= a.out_split) ? out2 + (o - a.out_split) : out + o;
                                    *dst = make_float2(x[k2].x, -x[k2].y);
                                }
                            }
                        }
                    }
                }
                __syncwarp();
            }
            parked = 0;
            sync_t();  // the parked spectra may be overwritten
        }
        PROF({ long long n_ = clock64(); tp[4] += n_ - tc; tc = n_; })
        // ---- hand the stage back to the front-end warps ---------------------------------------------------------------
        __syncwarp();
        if (lane == 0) {
            uint32_t left;
            asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(left) : "r"(left_cnt + (uint32_t)(gb & 1) * 4) : "memory");
            if (left % T_WARPS == T_WARPS - 1) {
                // the last transform warp to leave the stage: if the block after next is a stream's first, its kept rows start now
                int b2 = b + 2, so2 = so;
                while (b2 >= B) {
                    b2 -= B;
                    ++so2;
                }
                if (b2 == 0 && so2 < n_my) copy_kept(so2, gb + 2);
            }
            mb_arrive(bar_empty + (uint32_t)(gb & 1) * 8);
        }
    }
    PROF(if (tid == 0) for (int q = 0; q < 5; ++q) g_fused_prof[blockIdx.x * 16 + 9 + q] = tp[q];)
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
namespace {

using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                              const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn fused_encode_fn() {
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

template <int FW, int D, int NB> size_t fused_smem(int P, int Lmax) {
    const FusedGeom geo = fused_geom(P);
    size_t b = 2 * (size_t)STAGE_BYTES + TW_BYTES;
    b += ((size_t)Lmax * PITCH + 127) / 128 * 128;
    b += ((size_t)NB * YS_STRIDE * 8 + 127) / 128 * 128;
    b += (size_t)FW * D * geo.slot_stride;
    b += ((size_t)FW * P * 8 + 127) / 128 * 128;
    b += 32 + (size_t)FW * D * 8 + 64;
    return b;
}

template <int FW, int D, int NB, bool SHARED_IN>
cudaError_t launch_cfg(int n_streams, const FusedArgs& a, const CUtensorMap& tm, int sm_count, cudaStream_t st) {
    const size_t smem = fused_smem<FW, D, NB>(a.P, a.Lmax);
    if (smem > (size_t)227 * 1024) return cudaErrorInvalidConfiguration;
    const int grid = std::min(n_streams, sm_count);
    void (*kern)(const CUtensorMap, const FusedArgs, const int);
    // one instantiation per decimation factor: the front end's step loop must be unrolled completely for its coefficient
    // loads to go through the uniform datapath (with a run-time loop they are vector LDC loads and the kernel is slower
    // than k_front + k_poly2).  Common SDR ratios: 2.4 MS/s, 1.92 MS/s, 960 kS/s -> 48 kS/s.
    switch (a.P) {
        case 50: kern = a.nco ? k_fused<FW, D, NB, true, 50, SHARED_IN> : k_fused<FW, D, NB, false, 50, SHARED_IN>; break;
        case 40: kern = a.nco ? k_fused<FW, D, NB, true, 40, SHARED_IN> : k_fused<FW, D, NB, false, 40, SHARED_IN>; break;
        case 20: kern = a.nco ? k_fused<FW, D, NB, true, 20, SHARED_IN> : k_fused<FW, D, NB, false, 20, SHARED_IN>; break;
        default: return cudaErrorNotSupported;
    }
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, T_THREADS + 32 * FW, smem, st>>>(tm, a, n_streams);
#ifdef RR_FUSED_PROF
    static int calls = 0;
    static int at = std::getenv("RR_FUSED_PROF_CALL") ? std::atoi(std::getenv("RR_FUSED_PROF_CALL")) : 12;
    if (++calls == at) {
        cudaDeviceSynchronize();
        long long h[256 * 16];
        cudaMemcpyFromSymbol(h, g_fused_prof, sizeof h);
        for (int c : {0, 100})
            fprintf(stderr,
                    "cta %d n_out %d F0: tile-head %lld ring-wait %lld steps %lld fence+sync %lld issue %lld empty-wait %lld finalize %lld stream-setup %lld | total %lld"
                    " || T0: pre %lld wait-full %lld fwd+prod %lld sum+park %lld inverse %lld\n",
                    c, a.n_out, h[c * 16], h[c * 16 + 1], h[c * 16 + 2], h[c * 16 + 3], h[c * 16 + 4], h[c * 16 + 5], h[c * 16 + 6], h[c * 16 + 7], h[c * 16 + 8], h[c * 16 + 9],
                    h[c * 16 + 10], h[c * 16 + 11], h[c * 16 + 12], h[c * 16 + 13]);
    }
#endif
    return cudaGetLastError();
}

}  // namespace

int fused_coef_slots() { return kFusedSlots; }

bool fused_supported(int rank_pad, long long P, int Lmax) {
    if (rank_pad != FRK || !(P == 50 || P == 40 || P == 20) || fused_encode_fn() == nullptr) return false;  // launch_cfg's instantiations
    if (Lmax < 1 || FK - 1 - Lmax < 128 || Lmax > 383) return false;
    if ((P / 2) * 2 * FRK > kFusedSlotFloats) return false;
    return fused_smem<7, 2, 5>((int)P, Lmax) <= (size_t)227 * 1024;
}

cudaError_t fused_upload_coef(int slot, const float* acoef, int P, cudaStream_t st) {
    if (slot < 0 || slot >= kFusedSlots) return cudaErrorInvalidValue;
    const size_t n = (size_t)(P / 2) * 2 * FRK;
    if (n > (size_t)kFusedSlotFloats) return cudaErrorInvalidValue;
    return cudaMemcpyToSymbolAsync(c_fcoef, acoef, n * sizeof(float), (size_t)slot * kFusedSlotFloats * sizeof(float), cudaMemcpyHostToDevice, st);
}

cudaError_t launch_fused(int n_streams, const FusedArgs& a0, bool shared, int sm_count, cudaStream_t st) {
    EncodeFn enc = fused_encode_fn();
    if (!enc) return cudaErrorNotSupported;
    FusedArgs a = a0;
    a.coef_off4 = a.coef_slot * (kFusedSlotFloats / 4);
    // the kept rows of a stream enter the stage by one bulk copy: 16-byte aligned source
    if ((uintptr_t)a.ukeep_in % 16 != 0 || (n_streams > 1 && a.ukeep_in_stride % 2 != 0)) return cudaErrorInvalidValue;
    const FusedGeom geo = fused_geom(a.P);
    // the stream as overlapping rows of P samples: element (c0, i, s) = in[s*in_stride + c0 + i*P]; a box is half a
    // row wide and F_ROWS rows tall.  shared: one row that every stream reads (a zero stride cannot be encoded; the map
    // holds the row once and the kernel's shared form addresses it)
    if (shared != (n_streams > 1 && a.in_stride == 0)) return cudaErrorInvalidValue;
    CUtensorMap tm;
    const cuuint64_t dims[3] = {(cuuint64_t)a.len, (cuuint64_t)F_ROWS, (cuuint64_t)(shared ? 1 : n_streams)};
    const cuuint64_t sstride = n_streams > 1 && !shared ? (cuuint64_t)a.in_stride * 8 : (((cuuint64_t)a.len * 8 + 15) / 16) * 16;
    const cuuint64_t strides[2] = {(cuuint64_t)a.P * 8, sstride};
    const cuuint32_t box[3] = {(cuuint32_t)geo.hp, (cuuint32_t)F_ROWS, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<void*>(a.in), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    // configuration <front-end warps, ring depth, parked spectra>: seven front-end warps fill the register file next to the five
    // transform warps (12 warps x 168 registers) and were the fastest measured (RR_FUSED_CFG=1: six front-end warps, eight parked spectra)
    static int cfg = -1;
    if (cfg < 0) {
        cfg = 0;
        if (const char* e = std::getenv("RR_FUSED_CFG")) cfg = std::atoi(e);
    }
    if (shared) {
        switch (cfg) {
            case 1: return launch_cfg<6, 2, 8, true>(n_streams, a, tm, sm_count, st);
            default: return launch_cfg<7, 2, 5, true>(n_streams, a, tm, sm_count, st);
        }
    }
    switch (cfg) {
        case 1: return launch_cfg<6, 2, 8, false>(n_streams, a, tm, sm_count, st);
        default: return launch_cfg<7, 2, 5, false>(n_streams, a, tm, sm_count, st);
    }
}

}  // namespace rr
