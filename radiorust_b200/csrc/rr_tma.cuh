// TMA tensor maps of the pushed samples (k_poly2, k_front, k_fused) and the shared-memory / PTX wrappers that
// k_poly2 and k_fused have in common.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "rr_kernels.h"
#include "rr_pk.cuh"

namespace rr {

// ---- host: tensor maps ---------------------------------------------------------------------------------------------
using TmaEncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// the driver's cuTensorMapEncodeTiled, looked up once through the runtime (libcuda is not a link-time dependency);
// nullptr when the driver has none
inline TmaEncodeFn tma_encode_fn() {
    static TmaEncodeFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<TmaEncodeFn>(p);
    });
    return fn;
}

// a tiled map of UINT64 elements (one complex f32 sample each): dims[rank], byte strides of dimensions 1..rank-1,
// box[rank], element strides 1, no interleave, no swizzle, 128-byte L2 promotion, no out-of-bounds fill
inline bool tma_encode(CUtensorMap* tm, int rank, const void* base, const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box) {
    const TmaEncodeFn enc = tma_encode_fn();
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return enc && enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The stream dimension of an input map: n_streams rows in_stride samples apart, or (shared) the one row that every
// stream reads, mapped once (a zero stride cannot be encoded; the kernels' shared form addresses stream 0).  false
// when the input fails tma_input_ok or the shared flag does not match a zero stride.
struct TmaRows {
    cuuint64_t count;   // rows in the map
    cuuint64_t stride;  // bytes between them
};
inline bool tma_input_rows(const void* in, long long in_stride, long long len, int n_streams, bool shared, TmaRows* r) {
    if (shared != (n_streams > 1 && in_stride == 0) || !tma_input_ok(in, in_stride, len, n_streams, shared)) return false;
    r->count = shared ? 1 : (cuuint64_t)n_streams;
    r->stride = n_streams > 1 && !shared ? (cuuint64_t)in_stride * 8 : (((cuuint64_t)len * 8 + 15) / 16) * 16;
    return true;
}

// ---- device: shared-memory and PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ pc lds_pc(uint32_t addr) {
    pc r;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(addr));
    return r;
}
__device__ __forceinline__ void lds_pc2(uint32_t addr, pc& a, pc& b) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(b.x), "=f"(b.y) : "r"(addr));
}
__device__ __forceinline__ void sts_pc(uint32_t addr, pc a) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a.x), "f"(a.y) : "memory");
}
__device__ __forceinline__ void sts_pc2(uint32_t addr, pc a, pc b) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y) : "memory");
}
// read-only table load that stays where it is written (volatile asm keeps its place, so the load is
// in flight while the warp works on something else)
__device__ __forceinline__ void ldg_pc2(const float4* p, pc& a, pc& b) {
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(a.x), "=f"(a.y), "=f"(b.x), "=f"(b.y) : "l"(p));
}

// pass 1 of the 512-point forward transform of this thread's 32 inputs (rows t + 16*i1): radix-32
// butterfly, twiddles from table row `tw_row` (loaded two steps ahead of their use), element (t, k1)
// to row 33*t + k1 of the warp's strip (PITCH bytes per row)
template <int PITCH>
__device__ __forceinline__ void pass1_store(pc (&v)[32], uint32_t tw_row, uint32_t xch_wr) {
    pdft_regs<32, +1>(v);
    pc w[3][2];
    lds_pc2(tw_row, w[0][0], w[0][1]);
    lds_pc2(tw_row + 16, w[1][0], w[1][1]);
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        if (m + 2 < 16) lds_pc2(tw_row + (m + 2) * 16, w[(m + 2) % 3][0], w[(m + 2) % 3][1]);
        sts_pc(xch_wr + (2 * m) * PITCH, pcmul(v[2 * m], w[m % 3][0]));
        sts_pc(xch_wr + (2 * m + 1) * PITCH, pcmul(v[2 * m + 1], w[m % 3][1]));
    }
}

}  // namespace rr
