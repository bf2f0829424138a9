// Shared arithmetic of the decode-step kernels, so that a fused kernel and its stand-alone counterpart run the very same
// instruction sequence (bit-identical results).
#pragma once
#include "ptx.cuh"

namespace gb {

// Split-K partial sums.  Every load of a batch is issued before the first add: a plain `for (s < S) acc += ld(...)` loop is
// executed in order, so each iteration's add waits for its own load and a sum over S partials costs S serial L2 round trips
// (~0.7 us each on the decode critical path, between two weight-streaming GEMMs).  The adds still run in split order, so
// the result is bit-identical to the sequential loop.

// NP column groups at once: sum over the S partials ws[s][b][col[p] + {j, j+half}] of the token-major layout [S][B][N]
template <int NP>
__device__ __forceinline__ void splitk_pairs(const float* __restrict__ ws, int S, int B, int N, int b, const int (&col)[NP], int j,
                                             int half, float (&a1)[NP], float (&a2)[NP]) {
    constexpr int U = 4;
#pragma unroll
    for (int p = 0; p < NP; ++p) { a1[p] = 0.f; a2[p] = 0.f; }
    for (int s0 = 0; s0 < S; s0 += U) {
        float t1[U][NP], t2[U][NP];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int p = 0; p < NP; ++p)
                if (s0 + u < S) {
                    const float* row = ws + ((long long)(s0 + u) * B + b) * N + col[p] + j;
                    t1[u][p] = __ldcg(row);
                    t2[u][p] = __ldcg(row + half);
                }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int p = 0; p < NP; ++p)
                if (s0 + u < S) { a1[p] += t1[u][p]; a2[p] += t2[u][p]; }
    }
}

// sum over s < S of the float4 at p + s * stride (stride in floats), up to U loads in flight per pass
template <int U = 16>
__device__ __forceinline__ float4 splitk_sum4(const float* __restrict__ p, long long stride, int S) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s0 = 0; s0 < S; s0 += U) {
        float4 t[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (s0 + u < S) t[u] = __ldcg(reinterpret_cast<const float4*>(p + (long long)(s0 + u) * stride));
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (s0 + u < S) { a.x += t[u].x; a.y += t[u].y; a.z += t[u].z; a.w += t[u].w; }
    }
    return a;
}

// rotate-half RoPE of one (j, j+half) pair ($HF/models/llama/modeling_llama.py:138-168); inputs already rounded to bf16
__device__ __forceinline__ void rope_pair(float x1, float x2, float c, float sn, __nv_bfloat16& o1, __nv_bfloat16& o2) {
    // explicit mul + fma: every kernel that rotates (prefill GEMM epilogue, rope_kv_kernel, the decode kernels) must contract the
    // same way, or the last bit of a rotated value would depend on which of them produced it
    o1 = __float2bfloat16_rn(__fmaf_rn(x1, c, -__fmul_rn(x2, sn)));
    o2 = __float2bfloat16_rn(__fmaf_rn(x2, c, __fmul_rn(x1, sn)));
}

}  // namespace gb
