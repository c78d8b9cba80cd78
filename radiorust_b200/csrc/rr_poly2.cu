// k_poly2: the complex-f32 polyphase kernel of the fused chain
// FreqShifter -> Filter -> Downsampler (integer decimation, Q == 1, even P).
// It runs in two roles: on the output `u` of the rank-reduced front end
// (rr_front.cu; P = G = 10 branches, one round per block, no NCO: SINGLE) --
// that is the benchmarked path -- and on all P branches of the input itself
// when a filter does not factor to rank 10.
//
// Same algebra as k_poly (rr_poly.cuh: P branch transforms of K = 512 points, a
// multiply-accumulate against FFT_K(G[p]) and one inverse transform per block
// of V*P input samples), re-laid out for the issue-slot budget of an sm_100a
// SM -- k_poly is bound by instruction issue, not by HBM:
//
//   * every complex operation runs on the two-wide fp32 instructions
//     (rr_pk.cuh): half the issue slots for the same arithmetic;
//   * two passes instead of three: a radix-32 and two radix-16 butterflies per
//     thread, 16 threads per transform, ONE shared-memory exchange per
//     transform (conflict-free, constant offsets);
//   * the input tile of a round ([K rows][G branches] of the stream, rows P
//     samples apart) is brought in by one TMA tensor copy per round into a
//     two-stage mbarrier pipeline: no load instructions, no address arithmetic
//     and no load latency in the compute warps; the exchange reuses the
//     consumed tile in place;
//   * the NCO costs one complex multiply per sample: exp(j*w*(iP + p)) with
//     i = 16*i1 + t splits into exp(j*w*P*t), folded into the pass-1 twiddles,
//     and E[i1] * c_p (E[i1] = exp(j*w*16*P*i1), c_p the branch phasor), a
//     32-entry table per branch column that the column's 16 threads rebuild
//     for the next round while they work on the current one.
//
// Lane (t, column parity) of warp w works on branch column g = 2w + parity:
// pass 1 transforms rows t + 16*i1 of that column, pass 2 the bins k1 in
// {t, t+16}; it owns the 32 accumulators of bins t + 16*which + 32*k2.  The G partial spectra of a
// block are summed through shared memory once per block, parked, and inverted
// at the end by the same two-pass code (conjugate trick).
//
// A warp owns two branch columns end to end (both passes of both transforms),
// so a round needs no CTA-wide barrier: warps drift apart and one warp's
// shared-memory phases overlap another's arithmetic.  The warp that is last to
// hand a tile stage back starts the TMA copy of the round after next into it.
// One CTA = two independent halves (own stream, shared memory, mbarriers and
// named barrier): the register file is per SM sub-partition, so 10 warps of 168
// registers fit where two 5-warp CTAs would be rounded up.  Halves are
// persistent: each walks through (stream, group of blocks) units, the first tile
// of the next unit already in flight while the inverse transforms of the
// current one run.
//
// Blocks that reach before the pushed samples (into hist2, already mixed) take
// thread-local global loads instead of the TMA tile; a last block that would
// run past the pushed samples is moved back inside them.
//
// Reference semantics: transform.rs:333-348 (NCO), filters.rs:240-253
// (overlap-save filter), resampling.rs:103-121 (decimating FIR).
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>

#include "rr_kernels.h"
#include "rr_poly.cuh"
#include "rr_pk.cuh"
#include "rr_tma.cuh"

namespace rr {

namespace {

constexpr int K2 = 512;   // points per branch transform
constexpr int NT2 = 16;   // threads per transform
constexpr int ROWS_BOX = 256;

template <int G> struct P2Cfg {
    static_assert(G % 4 == 2, "a warp's two columns are conflict-free only when the tile pitch is an odd number of 16-byte units");
    static constexpr int NCW = G / 2;                // warps per half (two branch columns each)
    static constexpr int THREADS = 32 * NCW;         // threads per half
    static constexpr int PITCH = G * 8;              // bytes per tile row
    // A warp owns the 16-byte strip of its two columns in every row.  The exchange lives in the same
    // strip: element (t, k1) at row 33*t + k1 (rows 512..527 are spare), so that the pass-1 stores (lanes
    // t, fixed k1) and the pass-2 loads (lanes k1, fixed t) both walk 8 consecutive rows per quarter warp:
    // with an odd pitch/16 that is 8 distinct 16-byte bank groups, and every offset is an immediate.
    static constexpr int ROWS = 528;
    static constexpr int TILE_BYTES = K2 * PITCH;
    static constexpr int STAGE_BYTES = ROWS * PITCH;
    static_assert(STAGE_BYTES % 128 == 0, "TMA destination alignment");
    static constexpr int TW_UNITS = 17;              // 16-byte units per twiddle row t (16 + 1 pad)
    static constexpr int TW_BYTES = 16 * TW_UNITS * 16;
    static constexpr int E_BYTES = 400;              // E[32] | rowph[16] | rotG (+ pad to 16 bytes)
    static constexpr int ECP_BYTES = 16 * G * 16;    // one buffer of E[i1]*c_p: unit (m, g) = entries i1 = 2m, 2m+1 of column g
    static constexpr int YS_STRIDE = K2 + 1;         // parked spectrum stride (elements)
    static constexpr int OFF_STAGE = 0;
    static constexpr int OFF_TW = 2 * STAGE_BYTES;
    static constexpr int OFF_E = OFF_TW + TW_BYTES;
    static constexpr int OFF_ECP = OFF_E + E_BYTES;
    static constexpr int OFF_BAR = OFF_ECP + 2 * ECP_BYTES;  // full[2] (mbarriers), released[2] (counters)
    static constexpr int OFF_YS = OFF_BAR + 32;
    __host__ __device__ static size_t half_bytes(int nbpc) { return (((size_t)OFF_YS + (size_t)nbpc * YS_STRIDE * 8) + 127) / 128 * 128; }
    static size_t smem_bytes(int nbpc) { return 2 * half_bytes(nbpc); }
};

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
        "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ uint32_t atom_add_acqrel_shared(uint32_t addr, uint32_t v) {
    uint32_t old;
    asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(v) : "memory");
    return old;
}

}  // namespace

// One CTA = two independent halves (own stream, shared memory, mbarriers, named barrier).
// SINGLE: P <= G, one round per block (the low-rate part behind k_front): nothing is accumulated over
// rounds, the products go straight to the warp's strip and the block needs one barrier.
// SHARED_IN: every stream reads the same input row (the tensor map holds that one row, the copies address stream 0)
template <int G, bool HAS_NCO, bool SINGLE, bool SHARED_IN>
__global__ void __launch_bounds__(2 * P2Cfg<G>::THREADS, 1) k_poly2(const __grid_constant__ CUtensorMap tmap, const PolyArgs<float> a, const int n_streams) {
    using C = P2Cfg<G>;
    constexpr int THREADS = C::THREADS, PITCH = C::PITCH;
    const int half = threadIdx.x >= THREADS ? 1 : 0;
    const int tid = threadIdx.x - half * THREADS;
    const int warp = tid >> 5, lane = tid & 31;
    const int t = lane >> 1, gg = lane & 1;
    const int g = 2 * warp + gg;  // branch column of this lane
    // this half works through streams s_first, s_first + s_step, ...
    const int n_halves = a.halves == 1 ? 1 : 2;
    const int s_first = blockIdx.y * n_halves + half, s_step = gridDim.y * n_halves;
    if (s_first >= n_streams) return;  // the halves never meet at a CTA-wide barrier
    int s = s_first;
    auto sync_half = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(half + 1), "n"(THREADS) : "memory"); };

    extern __shared__ __align__(128) unsigned char smem_all[];
    unsigned char* smem = smem_all + (size_t)half * C::half_bytes(a.nbpc);
    const uint32_t sbase = smem_u32(smem);
    const uint32_t bar_full = sbase + C::OFF_BAR, cnt_rel = bar_full + 16;

    const int Pd = (int)a.P;
    const int NR = (Pd + G - 1) / G;
    const int len = (int)a.len, hist_len = (int)(2 * a.n);

    // window of block blk: element (i, p) sits at push offset boff + i*P + p.  "Interior" blocks lie
    // completely inside the pushed samples and are fed by TMA.  A block whose window would run past
    // the pushed samples is moved back by `d` rows so that it still lies inside them (its first d
    // outputs repeat the previous block's and are not stored).
    const int need = (K2 - 1) * Pd + NR * G;  // samples a tile sweep touches
    const bool sab = a.sab_blocks > 0;  // streams as blocks (short pushes)
    const int boff0 = (int)((a.I_lo - a.Lmax) * Pd - a.J0 - Pd);  // window start of block 0
    // block blk of a run of streams: real stream blk / rb within the run, its block blk % rb
    const int rb = sab ? max(1, a.sab_rb) : 1;
    auto blk_stream = [&](int blk) -> int { return sab ? blk / rb : 0; };
    auto blk_block = [&](int blk) -> int { return sab ? blk % rb : blk; };
    auto blk_start = [&](int blk) -> int {  // window start without any shift
        return boff0 + blk_stream(blk) * (int)a.sab_in_step + blk_block(blk) * a.V * Pd;
    };
    // only the last block can run past the end; block 0 has no predecessor to cover skipped outputs
    int last_shift = 0;
    {
        const int blk = a.n_blocks - 1;
        const int boff = blk_start(blk);
        if (blk > 0 && boff + need > len) {
            const int d = (boff + need - len + Pd - 1) / Pd;
            const long long Ibase = a.I_lo + (long long)blk_block(blk) * a.V - a.Lmax;
            // with Q == 1 the l = -1 slot of every branch filter is empty, so row K-1 is a valid output too:
            // the moved block may use it to reach m_hi
            if (d < a.V && boff - d * Pd >= 0 && a.m_hi - (Ibase - d) <= K2 - 1) last_shift = d;
        }
    }
    auto block_shift = [&](int blk) -> int { return blk == a.n_blocks - 1 ? last_shift : 0; };
    auto block_off = [&](int blk) -> int { return blk_start(blk) - block_shift(blk) * Pd; };
    auto is_interior = [&](int boff) -> bool { return boff >= 0 && boff + need <= len; };
    // the tile of round Rg of the group of stream `ss` that starts at block blk_first (nothing for edge blocks)
    auto issue_tile = [&](int ss, int blk_first, int blk_end, int Rg) {
        const int blk = blk_first + Rg / NR;
        if (blk >= blk_end) return;
        const int boff = block_off(blk);
        if (!is_interior(boff)) return;
        const int stage = Rg & 1;
        const uint32_t bar = bar_full + stage * 8;
        const uint32_t dst = sbase + C::OFF_STAGE + stage * C::STAGE_BYTES;
        mbar_expect_tx(bar, C::TILE_BYTES);
        if (SINGLE && Pd == G) {
            // P == G: the K rows of the tile are one contiguous run of the stream (16-byte aligned: boff is a
            // multiple of G = 10 samples, the stream stride is even)
            const float2* src = reinterpret_cast<const float2*>(a.in) + (long long)ss * a.in_stride + boff;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                         "r"((uint32_t)C::TILE_BYTES), "r"(bar)
                         : "memory");
        } else {
            tma_load_4d(dst, &tmap, bar, boff + (Rg % NR) * G, 0, 0, SHARED_IN ? 0 : ss);
        }
    };

    const uint32_t e_tab = sbase + C::OFF_E;
    const uint32_t ecp = sbase + C::OFF_ECP;
    const uint32_t tw_row = sbase + C::OFF_TW + t * (C::TW_UNITS * 16);
    // strip offsets inside a stage: tile row t, exchange row 33*t (stores), exchange row t (loads)
    const uint32_t tile_rd = t * PITCH + g * 8;
    const uint32_t xch_wr = 33 * t * PITCH + g * 8;
    const uint32_t xch_rd = t * PITCH + g * 8;
    float2* ysave = reinterpret_cast<float2*>(smem + C::OFF_YS);

    const float4* __restrict__ gtab = reinterpret_cast<const float4*>(a.gtab);
    uint32_t phase = 0;  // bit `stage`: parity of the next TMA completion to wait for

    // work units of this half: (stream, group of nbpc blocks), streams s_first, s_first + s_step, ...
    const int n_units = ((n_streams - s_first + s_step - 1) / s_step) * a.ngrp;
    auto unit_blocks = [&](int u, int* b0, int* b1) {
        *b0 = (blockIdx.x * a.ngrp + (u % a.ngrp)) * a.nbpc;
        *b1 = min(*b0 + a.nbpc, a.n_blocks);
    };
    // next unit after u that has blocks (n_units if none)
    auto next_unit = [&](int u) -> int {
        for (int v = u + 1; v < n_units; ++v) {
            int b0, b1;
            unit_blocks(v, &b0, &b1);
            if (b0 < b1) return v;
        }
        return n_units;
    };
    bool prefetched = false;  // (thread 0) the first two tiles of the current unit are already on their way

    for (int u = next_unit(-1); u < n_units; u = next_unit(u)) {
    s = s_first + (u / a.ngrp) * s_step;
    const bool new_stream = (u % a.ngrp) == 0 || u == next_unit(-1);
    const float2* __restrict__ in = reinterpret_cast<const float2*>(a.in) + (long long)s * a.in_stride;
    const float2* __restrict__ hist_end = reinterpret_cast<const float2*>(a.hist2) + ((long long)s + 1) * 2 * a.n;
    float2* __restrict__ out = reinterpret_cast<float2*>(a.out) + (long long)s * a.out_stride;
    float2* __restrict__ out2 = a.out2 ? reinterpret_cast<float2*>(a.out2) + (long long)s * a.out2_stride : nullptr;

    // ---- NCO constants, tables -------------------------------------------------------------
    uint32_t denom = 1, numer_abs = 0, idx0 = 0;
    int sign = 0;
    float start = 0.f;
    pc rotG(1.f, 0.f);
    if (HAS_NCO) {
        const NcoStream ns = a.nco[s];
        denom = ns.denom;
        numer_abs = ns.numer_abs;
        sign = ns.sign;
        idx0 = ns.idx;
        start = (float)ns.start_phase;
    }
    if ((HAS_NCO && new_stream) || u == next_unit(-1)) {  // the tables depend on the stream only through its NCO
        float2* et = reinterpret_cast<float2*>(smem + C::OFF_E);  // E[32] | rowph[16] | rotG
        if (tid < 49) {
            cx<float> r(1.f, 0.f);
            const long long d = tid < 32 ? (long long)16 * Pd * tid : (tid < 48 ? (long long)Pd * (tid - 32) : (long long)G);
            if (HAS_NCO) r = nco_rotation<float>(d, numer_abs, denom, sign);
            et[tid] = make_float2(r.x, r.y);
        }
        if (tid == 64 && u == next_unit(-1)) {
            mbar_init(bar_full, 1);
            mbar_init(bar_full + 8, 1);
            *reinterpret_cast<uint2*>(smem + C::OFF_BAR + 16) = make_uint2(0u, 0u);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        // pass-1 twiddles W_K^(t*k1) (the NCO's row part exp(j*w*P*t) is multiplied in below)
        const float2* __restrict__ twK = reinterpret_cast<const float2*>(a.twK);
        float2 w[(K2 + THREADS - 1) / THREADS];
#pragma unroll
        for (int i = 0; i < (K2 + THREADS - 1) / THREADS; ++i) {
            const int e = tid + i * THREADS;
            if (e < K2) w[i] = twK[((e >> 5) * (e & 31)) & (K2 - 1)];
        }
        sync_half();
#pragma unroll
        for (int i = 0; i < (K2 + THREADS - 1) / THREADS; ++i) {
            const int e = tid + i * THREADS;
            if (e < K2) {
                const int tr = e >> 5, k1 = e & 31;
                const float2 rp = et[32 + tr];
                const int off = (tr * C::TW_UNITS + (k1 >> 1)) * 16 + (k1 & 1) * 8;
                *reinterpret_cast<float2*>(smem + C::OFF_TW + off) = make_float2(w[i].x * rp.x - w[i].y * rp.y, w[i].x * rp.y + w[i].y * rp.x);
            }
        }
        sync_half();
    }
    if (HAS_NCO) rotG = lds_pc(e_tab + 48 * 8);
    const pc rowph = lds_pc(e_tab + (32 + t) * 8);
    // this lane's two entries of the E table (it maintains entries 2t, 2t+1 of its column's E*c_p)
    pc e_mine0(1.f, 0.f), e_mine1(1.f, 0.f);
    if (HAS_NCO) lds_pc2(e_tab + (2 * t) * 8, e_mine0, e_mine1);
    const uint32_t ecp_wr = ecp + (t * G + g) * 16;
    const uint32_t ecp_rd = ecp + g * 16;

    // hand stage (R & 1) back after round R of the group: the warp that completes the count starts the
    // TMA copy of round R + 2 into it
    auto release_stage = [&](int gb0, int gb1, int R) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            const uint32_t old = atom_add_acqrel_shared(cnt_rel + (R & 1) * 4, 1u);
            if (old % C::NCW == C::NCW - 1) issue_tile(s, gb0, gb1, R + 2);
        }
    };

    {
        int blk0, blk1;
        unit_blocks(u, &blk0, &blk1);
        if (tid == 0 && !prefetched) {
            issue_tile(s, blk0, blk1, 0);
            issue_tile(s, blk0, blk1, 1);
        }
        int R = 0;  // rounds of this group

        for (int blk = blk0; blk < blk1; ++blk) {
            const int boff = block_off(blk);
            const bool interior = is_interior(boff);

            pc cp(1.f, 0.f);  // NCO phasor of sample (i = 0, p = r*G + g) of this block, r = next round to prepare
            if (HAS_NCO) {
                if (lane < 2) {  // one evaluation per column
                    long long k0 = ((long long)idx0 + boff + g) % (long long)denom;
                    if (k0 < 0) k0 += denom;
                    const cx<float> c = nco_phasor<float>(mulmod_u32(numer_abs, (uint32_t)k0, denom), denom, sign, start);
                    cp = pc(c.x, c.y);
                }
                cp.x = __shfl_sync(0xffffffffu, cp.x, gg);
                cp.y = __shfl_sync(0xffffffffu, cp.y, gg);
                // E*c_p of round 0 (the buffer's last readers were this warp's own lanes, two rounds ago)
                sts_pc2(ecp_wr + (R & 1) * C::ECP_BYTES, pcmul(e_mine0, cp), pcmul(e_mine1, cp));
                __syncwarp();
            }
            pc acc[32];
            if (!SINGLE) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = pc(0.f, 0.f);
            }

            for (int r = 0; r < NR; ++r, ++R) {
                const int stage = R & 1;
                const uint32_t stg = sbase + C::OFF_STAGE + stage * C::STAGE_BYTES;
                const uint32_t esrc = ecp_rd + stage * C::ECP_BYTES;
                pc v[32];
                if (interior) {
                    mbar_wait(bar_full + stage * 8, (phase >> stage) & 1);
                    phase ^= 1u << stage;
                    const uint32_t src = stg + tile_rd;
#pragma unroll
                    for (int m = 0; m < 16; ++m) {
                        pc e0, e1;
                        if (HAS_NCO) lds_pc2(esrc + m * (G * 16), e0, e1);
                        v[2 * m] = lds_pc(src + (2 * m) * (16 * PITCH));
                        v[2 * m + 1] = lds_pc(src + (2 * m + 1) * (16 * PITCH));
                        if (HAS_NCO) {
                            v[2 * m] = pcmul(v[2 * m], e0);
                            v[2 * m + 1] = pcmul(v[2 * m + 1], e1);
                        }
                    }
                } else {
                    // thread-local loads (all issued first, predicated); history samples are already mixed:
                    // for them only the row part that the twiddles will apply is cancelled
                    // (the offsets are made opaque so that the compiler does not carry 32 induction variables of
                    // this rarely taken branch through the round loop)
                    int r_o = r, boff_o = boff;
                    asm volatile("" : "+r"(r_o), "+r"(boff_o));
                    const int p = r_o * G + g;
                    const int pos0 = boff_o + t * Pd + p;
                    const int step = 16 * Pd;
                    const unsigned span = (unsigned)(len + hist_len);
#pragma unroll
                    for (int i1 = 0; i1 < 32; ++i1) {
                        const int pos = pos0 + i1 * step;
                        const bool ok = p < Pd && (unsigned)(pos + hist_len) < span;
                        const float2* ptr = (pos >= 0 ? in : hist_end) + pos;
                        float2 q = make_float2(0.f, 0.f);
                        if (ok) q = __ldg(ptr);
                        v[i1] = pc(q.x, q.y);
                    }
                    if (HAS_NCO) {
                        const pc hc(rowph.x, -rowph.y);
#pragma unroll
                        for (int m = 0; m < 16; ++m) {
                            pc e0, e1;
                            lds_pc2(esrc + m * (G * 16), e0, e1);
                            v[2 * m] = pcmul(v[2 * m], (pos0 + (2 * m) * step) >= 0 ? e0 : hc);
                            v[2 * m + 1] = pcmul(v[2 * m + 1], (pos0 + (2 * m + 1) * step) >= 0 ? e1 : hc);
                        }
                    }
                }
                if (HAS_NCO) {
                    // next round's E*c_p (other buffer: its readers were this warp's lanes, a round ago)
                    cp = pcmul(cp, rotG);
                    if (r + 1 < NR) sts_pc2(ecp_wr + (stage ^ 1) * C::ECP_BYTES, pcmul(e_mine0, cp), pcmul(e_mine1, cp));
                }
                __syncwarp();  // the strip's tile rows are consumed by every lane before any lane overwrites them
                pass1_store<PITCH>(v, tw_row, stg + xch_wr);

                // table entries of this round: [r][which][jj][tid] (two bins each)
                const float4* gp = gtab + ((long long)r * 16) * THREADS + tid;
                pc h[16];
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) ldg_pc2(gp + jj * THREADS, h[2 * jj], h[2 * jj + 1]);
                __syncwarp();
#pragma unroll
                for (int which = 0; which < 2; ++which) {
                    pc x[16];
#pragma unroll
                    for (int tr = 0; tr < 16; ++tr) x[tr] = lds_pc(stg + xch_rd + (33 * tr + 16 * which) * PITCH);
                    pdft_regs<16, +1>(x);
                    if (which == 1 && r + 1 < NR) release_stage(blk0, blk1, R);  // the exchange is read: stage free
#pragma unroll
                    for (int k = 0; k < 16; ++k) acc[which * 16 + k] = SINGLE ? pcmul(x[k], h[k]) : pcfma(x[k], h[k], acc[which * 16 + k]);
                    if (which == 0) {
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj) ldg_pc2(gp + (8 + jj) * THREADS, h[2 * jj], h[2 * jj + 1]);
                    }
                }
            }

            // ---- sum the G partial spectra of this block, park the result; the block's last stage is
            //      the scratch area and is released afterwards ------------------------------------------
            if (SINGLE) {
                // the exchange of this warp's strip is consumed: park bin (j, t) of its two columns at row 16*j + t
                const uint32_t stg = sbase + C::OFF_STAGE + ((R - 1) & 1) * C::STAGE_BYTES;
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 32; ++j) sts_pc(stg + xch_rd + (16 * j) * PITCH, acc[j]);
                sync_half();
                float2* ys = ysave + (blk - blk0) * C::YS_STRIDE;
                for (int o = tid; o < K2; o += THREADS) {
                    const uint32_t src = stg + o * PITCH;  // row o: the G columns side by side
                    pc sum(0.f, 0.f);
#pragma unroll
                    for (int w = 0; w < C::NCW; ++w) {
                        pc u0, u1;
                        lds_pc2(src + w * 16, u0, u1);
                        sum = sum + u0;
                        sum = sum + u1;
                    }
                    const int j = o >> 4, tt = o & 15;
                    ys[tt + 16 * (j >> 4) + 32 * (j & 15)] = make_float2(sum.x, sum.y);
                }
                release_stage(blk0, blk1, R - 1);
            } else {
                const uint32_t stg = sbase + C::OFF_STAGE + ((R - 1) & 1) * C::STAGE_BYTES;
                sync_half();
#pragma unroll
                for (int j = 0; j < 32; ++j) sts_pc(stg + (j * THREADS + tid) * 8, acc[j]);
                sync_half();
                float2* ys = ysave + (blk - blk0) * C::YS_STRIDE;
                for (int o = tid; o < K2; o += THREADS) {
                    const int j = o >> 4, tt = o & 15;
                    const uint32_t src = stg + (j * THREADS + 2 * tt) * 8;
                    pc sum(0.f, 0.f);
#pragma unroll
                    for (int w = 0; w < C::NCW; ++w) {
                        pc u0, u1;
                        lds_pc2(src + w * 256, u0, u1);
                        sum = sum + u0;
                        sum = sum + u1;
                    }
                    const int bin = tt + 16 * (j >> 4) + 32 * (j & 15);
                    ys[bin] = make_float2(sum.x, sum.y);
                }
                release_stage(blk0, blk1, R - 1);
            }
        }
        sync_half();
        // both stages are free now: the next unit's first tile goes into stage 0 while the inverse transforms
        // exchange through stage 1
        const int u_next = next_unit(u);
        int nb0 = 0, nb1 = 0;
        if (u_next < n_units) unit_blocks(u_next, &nb0, &nb1);
        const int s_next = s_first + (u_next / a.ngrp) * s_step;
        if (tid == 0) {
            prefetched = u_next < n_units;
            if (prefetched) issue_tile(s_next, nb0, nb1, 0);
        }

        // ---- inverse transforms: branch column g takes job g (one parked block spectrum) -------------
        const int njobs = blk1 - blk0;
        for (int j0 = 0; j0 < njobs; j0 += G) {
            if (j0 + 2 * warp >= njobs) continue;  // neither column of this warp has a job (warp-uniform)
            const int job = j0 + g;
            const bool active = job < njobs;
            const uint32_t stg = sbase + C::OFF_STAGE + C::STAGE_BYTES;
            pc v[32];
            const float2* ys = ysave + (active ? job : 0) * C::YS_STRIDE;
            // conj in, conj out = inverse transform; the table's NCO row part is cancelled on the way in
            const pc hc(rowph.x, -rowph.y);
#pragma unroll
            for (int i1 = 0; i1 < 32; ++i1) {
                const float2 q = ys[t + 16 * i1];
                v[i1] = active ? pcmul(pc(q.x, -q.y), hc) : pc(0.f, 0.f);
            }
            pass1_store<PITCH>(v, tw_row, stg + xch_wr);
            __syncwarp();
            const int blk = blk0 + (active ? job : 0);
            const int d = block_shift(blk);
            const long long Ibase = a.I_lo + (long long)blk_block(blk) * a.V - a.Lmax - d;
            // streams as blocks: the block belongs to real stream s*(sab_blocks/rb) + blk/rb with its own destinations
            const int rs = blk_stream(blk);
            const bool exists = !sab || (long long)s * (a.sab_blocks / rb) + rs < a.sab_streams;
            float2* outb = sab ? out + (long long)rs * a.sab_out_step : out;
            float2* out2b = (sab && out2 != nullptr) ? out2 + (long long)rs * a.sab_out2_step : out2;
#pragma unroll
            for (int which = 0; which < 2; ++which) {
                pc x[16];
#pragma unroll
                for (int tr = 0; tr < 16; ++tr) x[tr] = lds_pc(stg + xch_rd + (33 * tr + 16 * which) * PITCH);
                pdft_regs<16, +1>(x);
                if (active) {
#pragma unroll
                    for (int k2 = 0; k2 < 16; ++k2) {
                        const int i = t + 16 * which + 32 * k2;
                        if (i >= a.Lmax + d && i < a.Lmax + a.V + (d > 0 ? 1 : 0)) {
                            const long long m = Ibase + i;  // Q == 1
                            if (m >= a.m_lo && m <= a.m_hi && exists) {
                                const long long o = m - a.m0 - 1;
                                float2* dst = (out2b != nullptr && o >= a.out_split) ? out2b + (o - a.out_split) : outb + o;
                                *dst = make_float2(x[k2].x, -x[k2].y);
                            }
                        }
                    }
                }
            }
            __syncwarp();
        }
        // the next unit's second tile goes into the stage the inverse just used
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        sync_half();
        if (tid == 0 && prefetched) issue_tile(s_next, nb0, nb1, 1);
    }
    }  // units
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
namespace {

template <int G>
cudaError_t launch_g(int n_streams, const PolyArgs<float>& a, const CUtensorMap& tm, bool shared, int sm_count, cudaStream_t st) {
    using C = P2Cfg<G>;
    const int halves = a.halves == 1 ? 1 : 2;
    const size_t smem = C::half_bytes(a.nbpc) * halves;
    const int per_cta = a.nbpc * (a.ngrp > 0 ? a.ngrp : 1);
    // one CTA per SM; a half walks through several streams when there are more stream pairs than SMs
    const unsigned gx = (unsigned)((a.n_blocks + per_cta - 1) / per_cta);
    unsigned gy = (unsigned)((n_streams + halves - 1) / halves);
    const int slots = sm_count * (halves == 1 ? 2 : 1);  // CTAs that can be resident at once
    if ((long long)gx * gy > slots) gy = (unsigned)std::max(1, std::min((int)gy, (slots + (int)gx - 1) / (int)gx));
    const dim3 grid(gx, gy);
    void (*kern)(const CUtensorMap, const PolyArgs<float>, const int);
    const bool single = a.P <= G;
    if (shared) {
        if (a.nco) kern = single ? k_poly2<G, true, true, true> : k_poly2<G, true, false, true>;
        else kern = single ? k_poly2<G, false, true, true> : k_poly2<G, false, false, true>;
    } else if (a.nco) {
        kern = single ? k_poly2<G, true, true, false> : k_poly2<G, true, false, false>;
    } else {
        kern = single ? k_poly2<G, false, true, false> : k_poly2<G, false, false, false>;
    }
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, halves * C::THREADS, smem, st>>>(tm, a, n_streams);
    return cudaGetLastError();
}

}  // namespace

int poly2_pick_G(long long P) {
    // branches per round: even (TMA rows are 16-byte multiples) and as few idle columns as possible
    int best = 0;
    double best_eff = 0.0;
    for (int G : {10}) {
        const double eff = (double)P / (double)(G * ((P + G - 1) / G));
        if (eff > best_eff + 1e-9) {
            best = G;
            best_eff = eff;
        }
    }
    return best_eff >= 0.5 ? best : 0;
}

bool poly2_supported(int K, long long P, long long Q) {
    return K == K2 && Q == 1 && P >= 2 && (P % 2) == 0 && poly2_pick_G(P) != 0 && tma_encode_fn() != nullptr;
}

size_t poly2_smem_bytes(int G, int nbpc) { return P2Cfg<10>::smem_bytes(nbpc); }

long long poly2_table_index(int G, int r, int g, int k) {
    const int threads = NT2 * G;  // compute threads per half
    const int k1 = k & 31, k2 = k >> 5;
    const int tt = k1 & 15, which = k1 >> 4;
    const int tid = (g >> 1) * 32 + 2 * tt + (g & 1);  // warp g/2, lane (t, column parity)
    return ((((long long)r * 2 + which) * 8 + (k2 >> 1)) * threads + tid) * 2 + (k2 & 1);
}

cudaError_t launch_poly2(int G, int n_streams, const PolyArgs<float>& a, bool shared, int sm_count, cudaStream_t st) {
    if (!tma_encode_fn()) return cudaErrorNotSupported;
    // the stream as overlapping rows: element (c0, i_lo, i_hi, s) = in[s*in_stride + c0 + (i_lo + 256*i_hi)*P].  The
    // low-rate part on u, streams-as-blocks form included, reads per-stream rows.
    TmaRows rows;
    if (!tma_input_rows(a.in, a.in_stride, a.len, n_streams, shared, &rows)) return cudaErrorInvalidValue;
    CUtensorMap tm;
    const cuuint64_t dims[4] = {(cuuint64_t)a.len, (cuuint64_t)ROWS_BOX, (cuuint64_t)(K2 / ROWS_BOX), rows.count};
    const cuuint64_t strides[3] = {(cuuint64_t)a.P * 8, (cuuint64_t)a.P * 8 * ROWS_BOX, rows.stride};
    const cuuint32_t box[4] = {(cuuint32_t)G, (cuuint32_t)ROWS_BOX, (cuuint32_t)(K2 / ROWS_BOX), 1};
    if (!tma_encode(&tm, 4, a.in, dims, strides, box)) return cudaErrorInvalidValue;
    if (G == 10) return launch_g<10>(n_streams, a, tm, shared, sm_count, st);
    return cudaErrorInvalidValue;
}

}  // namespace rr
