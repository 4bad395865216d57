// canonical.cuh — the canonical score arithmetic shared by the exact kernels (knn_exact.cu, kmeans.cu).
// Bit-for-bit what oracle/faiss_flat.c `orc_dot_canonical` / `orc_l2_canonical` compute: element i is accumulated by lane
// (i>>2)&31 in increasing i with fp64 fma; the 32 partials are combined by a 16,8,4,2,1 xor-butterfly; the double is rounded
// once to fp32.
#pragma once
#include "common.cuh"

namespace b2 {
namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double butterfly_sum(double v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
    return v;
}

// exact float32 value of element i of a B2_F32 / B2_BF16 / B2_F16 array (both 2-byte types widen exactly)
__device__ __forceinline__ float elem_f32(const void* base, int dtype, size_t i) {
    if (dtype == B2_F32) return reinterpret_cast<const float*>(base)[i];
    if (dtype == B2_F16) return __half2float(reinterpret_cast<const __half*>(base)[i]);
    return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[i]);
}

// the four fp16 values packed in two 32-bit words, widened
__device__ __forceinline__ void f16x4_to_f32(uint2 t, float (&o)[4]) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}

// 4 consecutive elements of group g of a row (zero beyond d). `vec` = row start is 4-element aligned.
__device__ __forceinline__ void load_group(const void* row, int dtype, int g, int d, bool vec, float (&o)[4]) {
    const int i0 = g * 4;
    if (vec) {
        if (dtype == B2_F32) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(row) + g);
            o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
        } else if (dtype == B2_F16) {
            f16x4_to_f32(__ldg(reinterpret_cast<const uint2*>(row) + g), o);
        } else {
            const uint2 t = __ldg(reinterpret_cast<const uint2*>(row) + g);
            o[0] = __uint_as_float(t.x << 16);
            o[1] = __uint_as_float(t.x & 0xffff0000u);
            o[2] = __uint_as_float(t.y << 16);
            o[3] = __uint_as_float(t.y & 0xffff0000u);
        }
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = (i0 + e < d) ? elem_f32(row, dtype, (size_t)(i0 + e)) : 0.f;
    }
}

// canonical partial (this lane's share) of <q, x> or ||q - x||^2; q lives in shared memory as fp32
template <bool IS_L2>
__device__ __forceinline__ double canonical_partial(const float* q_s, const void* row, int dtype, int d, bool vec, int lane) {
    double acc = 0.0;
    const int ngroups = (d + 3) >> 2;
    for (int g = lane; g < ngroups; g += 32) {
        float x[4];
        load_group(row, dtype, g, d, vec, x);
        const float4 q4 = *reinterpret_cast<const float4*>(q_s + 4 * g);
        const float qq[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            if (IS_L2) {
                const double diff = (double)qq[e] - (double)x[e];
                acc = fma(diff, diff, acc);
            } else {
                acc = fma((double)qq[e], (double)x[e], acc);
            }
        }
    }
    return acc;
}

}  // namespace
}  // namespace b2
