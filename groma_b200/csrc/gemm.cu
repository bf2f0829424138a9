// Host launcher for the tcgen05 GEMM / implicit-GEMM conv and the split-K reduce epilogue.
// C ABI: see include/groma_b200.h (groma_gemm_bf16, groma_splitk_reduce).
#include "gemm_tcgen05.cuh"
#include "capi_common.h"

namespace gb {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    return fn;
}

// 2D bf16 row-major tensor [rows, cols] with row stride ld (elements); box = {64 cols, box_rows}; 128B swizzle.
static int make_tma_2d(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return GROMA_ERR_DRIVER;
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 2};
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? GROMA_OK : GROMA_ERR_TMA_ENCODE;
}

static int g_num_sms = 0;
static int num_sms() {
    if (!g_num_sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    }
    return g_num_sms;
}

// 2-CTA (cta_group::2) launch: clusters of two CTAs, each cluster owns 256 x 256 output tiles
static int launch_gemm_2cta(const GemmParams& p, cudaStream_t stream) {
    using Cfg = GemmCfg<256, 2>;
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess)
            return GROMA_ERR_CUDA;
        attr_set = true;
    }
    const int m_tiles = (p.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM);
    const int n_tiles = (p.N + 255) / 256;
    const int work = m_tiles * n_tiles;
    int clusters = num_sms() / 2;
    if (work < clusters) clusters = work;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(clusters * 2); cfg.blockDim = dim3(Cfg::THREADS); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, gemm_bf16_tcgen05_kernel<256, 2>, p) == cudaSuccess ? GROMA_OK : GROMA_ERR_CUDA;
}

template <int BN>
static int launch_gemm(const GemmParams& p, cudaStream_t stream) {
    using Cfg = GemmCfg<BN>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<BN, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             Cfg::SMEM_BYTES);
        if (e != cudaSuccess) return GROMA_ERR_CUDA;
        attr_set = true;
    }
    const int m_tiles = (p.M + GEMM_BM - 1) / GEMM_BM;
    const int n_tiles = (p.N + BN - 1) / BN;
    const int work = m_tiles * n_tiles * p.split_k;
    // BN = 16 (decode swap-AB): 4-stage ring, two CTAs per SM -- one CTA's tile epilogue / tile switch overlaps the other's
    // streaming (measured: GEMM-only decode graph 2.34 -> 2.25 ms vs one 8-stage CTA per SM).  GromaEngine._decode_splits
    // sizes the decode split-K factors for these 2 CTAs per SM: change both together.
    const int slots = num_sms() * (BN == 16 ? 2 : 1);
    const int grid = work < slots ? work : slots;
    if (p.flags & GF_PDL) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(Cfg::THREADS); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, gemm_bf16_tcgen05_kernel<BN, 1>, p) == cudaSuccess ? GROMA_OK : GROMA_ERR_CUDA;
    }
    gemm_bf16_tcgen05_kernel<BN, 1><<<grid, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(p);
    return cudaGetLastError() == cudaSuccess ? GROMA_OK : GROMA_ERR_CUDA;
}

// ------------------------------------------------------------------ split-K reduce + epilogue
// out[m,n] = epi(sum_s ws[s][m][n]); same epilogue chain as the GEMM kernel.  SWIGLU pairs columns.
__global__ void splitk_reduce_kernel(const float* __restrict__ ws, int splits, int M, int N, int act, int flags,
                                     const float* __restrict__ bias, const float* __restrict__ gamma,
                                     const __nv_bfloat16* __restrict__ residual, void* __restrict__ out, long long ld_m,
                                     long long ld_n) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const bool bias_m0 = flags & GF_BIAS_ALONG_M;
    const long long total = (act == ACT_SWIGLU) ? (bias_m0 ? (long long)(M / 2) * N : (long long)M * (N / 2)) : (long long)M * N;
    const bool bias_m = flags & GF_BIAS_ALONG_M;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        if (act == ACT_SWIGLU && bias_m) {
            // swap-AB layout: ws[s][M = 2*I rows (gate_j, up_j interleaved)][N = tokens] -> out[token, j]
            const int t = i % N;
            const long long j = i / N;  // i in [0, (M/2)*N)
            float g = 0.f, u = 0.f;
            for (int s2 = 0; s2 < splits; ++s2) {
                g += ws[((long long)s2 * M + 2 * j) * N + t];
                u += ws[((long long)s2 * M + 2 * j + 1) * N + t];
            }
            reinterpret_cast<__nv_bfloat16*>(out)[j * ld_m + t * ld_n] = __float2bfloat16_rn(silu(g) * u);
            continue;
        }
        if (act == ACT_SWIGLU) {
            const int NO = N / 2;
            const int m = i / NO, j = i - (long long)m * NO;
            float g = 0.f, u = 0.f;
            for (int s = 0; s < splits; ++s) {
                const float2 v = *reinterpret_cast<const float2*>(ws + ((long long)s * M + m) * N + 2 * j);
                g += v.x;
                u += v.y;
            }
            if (bias) { g += bias[2 * j]; u += bias[2 * j + 1]; }
            reinterpret_cast<__nv_bfloat16*>(out)[m * ld_m + j * ld_n] = __float2bfloat16_rn(silu(g) * u);
            continue;
        }
        const int m = i / N, n = i - (long long)m * N;
        float v = 0.f;
        for (int s0 = 0; s0 < splits; s0 += 8) {   // all partial loads of a batch in flight before the first add (same add order)
            float t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) if (s0 + u < splits) t[u] = ws[((long long)(s0 + u) * M + m) * N + n];
#pragma unroll
            for (int u = 0; u < 8; ++u) if (s0 + u < splits) v += t[u];
        }
        if (bias) v += bias[bias_m ? m : n];
        v = apply_act(v, act);
        if (gamma) v *= gamma[bias_m ? m : n];
        const long long o = m * ld_m + n * ld_n;
        if (residual) v += __bfloat162float(residual[o]);
        if (flags & GF_OUT_F32) reinterpret_cast<float*>(out)[o] = v;
        else reinterpret_cast<__nv_bfloat16*>(out)[o] = __float2bfloat16_rn(v);
    }
}

}  // namespace gb

using namespace gb;

namespace {
struct RopeEpilogue {   // GF_ROPE_QKV operands (see GemmParams)
    const float* cos_t; const float* sin_t; void* cache_k; void* cache_v;
    int T, H, pos0; long long cap;
};
}  // namespace

static int32_t gemm_impl(const void* A, int64_t a_rows, int64_t lda, const void* B, int64_t b_rows,
                         int64_t ldb, int32_t M, int32_t N, int32_t K, int32_t num_taps,
                         const int32_t* a_row_off, void* out, int64_t ld_m, int64_t ld_n, int32_t flags,
                         int32_t act, const float* bias, const float* gamma, const void* residual,
                         float* ws, int32_t split_k, int32_t conv_hp, int32_t conv_wp,
                         int32_t block_n, void* stream, const RopeEpilogue* rope) {
    if (!A || !B || M <= 0 || N <= 0 || K <= 0) return GROMA_ERR_ARG;
    if (((flags & GF_ROPE_QKV) != 0) != (rope != nullptr)) return GROMA_ERR_ARG;
    if (num_taps < 1 || num_taps > GEMM_MAX_TAPS) return GROMA_ERR_ARG;
    if ((lda & 7) || (ldb & 7) || (reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15))
        return GROMA_ERR_ALIGN;
    if (split_k < 1) split_k = 1;
    if (split_k > 1 && !(flags & GF_PARTIAL)) return GROMA_ERR_ARG;
    if ((flags & GF_PARTIAL) && !ws) return GROMA_ERR_ARG;
    if (!(flags & GF_PARTIAL) && !out) return GROMA_ERR_ARG;
    if (act == ACT_SWIGLU && !(flags & GF_BIAS_ALONG_M) && (N & 1)) return GROMA_ERR_ARG;
    if (act == ACT_SWIGLU && (flags & GF_BIAS_ALONG_M) && (M & 1)) return GROMA_ERR_ARG;
    if (num_taps > 1 && (K % GEMM_BK) != 0) return GROMA_ERR_ARG;

    int bn = block_n;
    if (bn == 0) {
        // widest tile that still gives every SM work; small N gets the tile that fits it
        if (N <= 16) bn = 16;
        else if (N <= 32) bn = 32;
        else if (N <= 64) bn = 64;
        else {
            const long long m_tiles = (M + GEMM_BM - 1) / GEMM_BM;
            const long long t256 = m_tiles * ((N + 255) / 256) * split_k;
            bn = (N >= 256 && t256 >= num_sms()) ? 256 : 128;
            if (bn == 128 && m_tiles * ((N + 127) / 128) * split_k < num_sms() / 2 && N >= 128) bn = 64;
        }
    }
    GemmParams p;
    int rc = make_tma_2d(&p.tma_a, A, (uint64_t)a_rows, (uint64_t)K, (uint64_t)lda, GEMM_BM);
    if (rc) return rc;
    rc = make_tma_2d(&p.tma_b, B, (uint64_t)b_rows, (uint64_t)K * num_taps, (uint64_t)ldb, bn == 512 ? 128u : (uint32_t)bn);
    if (rc) return rc;
    p.M = M; p.N = N; p.K = K; p.num_taps = num_taps;
    for (int i = 0; i < GEMM_MAX_TAPS; ++i) p.a_row_off[i] = (a_row_off && i < num_taps) ? a_row_off[i] : 0;
    p.split_k = split_k; p.flags = flags; p.act = act;
    p.out = out; p.ld_m = ld_m; p.ld_n = ld_n;
    p.bias = bias; p.gamma = gamma; p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
    p.ws = ws; p.conv_hp = conv_hp; p.conv_wp = conv_wp;
    p.rope_cos = p.rope_sin = nullptr; p.rope_k = p.rope_v = nullptr; p.rope_T = 1; p.rope_H = 1; p.rope_pos0 = 0; p.rope_cap = 0;
    if (rope) {
        if (bn != 256 && bn != 512) return GROMA_ERR_UNSUPPORTED;   // one head (128 columns) per epilogue warp needs the 256-wide tile
        p.rope_cos = rope->cos_t; p.rope_sin = rope->sin_t;
        p.rope_k = reinterpret_cast<__nv_bfloat16*>(rope->cache_k); p.rope_v = reinterpret_cast<__nv_bfloat16*>(rope->cache_v);
        p.rope_T = rope->T; p.rope_H = rope->H; p.rope_pos0 = rope->pos0; p.rope_cap = rope->cap;
    }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (bn == 512) {   // block_n = 512 selects the 2-CTA (256 x 256 per cluster) kernel
        if (split_k != 1 || (flags & (GF_PARTIAL | GF_PDL))) return GROMA_ERR_ARG;
        return launch_gemm_2cta(p, st);
    }
    switch (bn) {
        case 16: return launch_gemm<16>(p, st);
        case 32: return launch_gemm<32>(p, st);
        case 64: return launch_gemm<64>(p, st);
        case 128: return launch_gemm<128>(p, st);
        case 256: return launch_gemm<256>(p, st);
        default: return GROMA_ERR_ARG;
    }
}

GROMA_API int32_t groma_gemm_bf16(const void* A, int64_t a_rows, int64_t lda, const void* B, int64_t b_rows,
                                   int64_t ldb, int32_t M, int32_t N, int32_t K, int32_t num_taps,
                                   const int32_t* a_row_off, void* out, int64_t ld_m, int64_t ld_n, int32_t flags,
                                   int32_t act, const float* bias, const float* gamma, const void* residual,
                                   float* ws, int32_t split_k, int32_t conv_hp, int32_t conv_wp,
                                   int32_t block_n, void* stream) {
    if (flags & GF_ROPE_QKV) return GROMA_ERR_ARG;   // that epilogue has its own entry point below
    return gemm_impl(A, a_rows, lda, B, b_rows, ldb, M, N, K, num_taps, a_row_off, out, ld_m, ld_n, flags, act, bias, gamma,
                     residual, ws, split_k, conv_hp, conv_wp, block_n, stream, nullptr);
}

// LLaMA attention input in one launch: x [B*T, K] @ Wqkv^T [3*H*128, K] with rotate-half RoPE on q/k and the KV-cache
// append done by the GEMM epilogue (replaces q_proj/k_proj/v_proj + apply_rotary_pos_emb + the cache torch.cat of
// $HF/models/llama/modeling_llama.py:199-246).  q_out [B*T, H*128]; cache_k/v [B, H, ctx_cap, 128]; token t of every
// sequence sits at position pos0 + t.  block_n: 256 (one CTA per tile) or 512 (cta_group::2 pair).
GROMA_API int32_t groma_gemm_qkv_rope(const void* x, int64_t ldx, const void* w_qkv, int64_t ldw, int32_t B, int32_t T,
                                       int32_t H, int32_t D, int32_t K, void* q_out, void* cache_k, void* cache_v,
                                       const float* cos_t, const float* sin_t, int32_t pos0, int64_t ctx_cap,
                                       int32_t block_n, void* stream) {
    if (!x || !w_qkv || !q_out || !cache_k || !cache_v || !cos_t || !sin_t) return GROMA_ERR_ARG;
    if (B <= 0 || T <= 0 || H <= 0 || K <= 0 || pos0 < 0 || (long long)pos0 + T > ctx_cap) return GROMA_ERR_ARG;
    if (D != 128 || (H & 1)) return GROMA_ERR_UNSUPPORTED;          // 3*H*128 must tile by 256 columns
    if (block_n != 256 && block_n != 512) return GROMA_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(q_out) | reinterpret_cast<uintptr_t>(cache_k) | reinterpret_cast<uintptr_t>(cache_v) |
         reinterpret_cast<uintptr_t>(cos_t) | reinterpret_cast<uintptr_t>(sin_t)) & 15) return GROMA_ERR_ALIGN;
    RopeEpilogue r{cos_t, sin_t, cache_k, cache_v, T, H, pos0, (long long)ctx_cap};
    const long long M = (long long)B * T;
    if (M > 0x7fffffffLL) return GROMA_ERR_ARG;
    return gemm_impl(x, M, ldx, w_qkv, 3LL * H * D, ldw, (int32_t)M, 3 * H * D, K, 1, nullptr, q_out, (int64_t)H * D, 1,
                     GF_ROPE_QKV, ACT_NONE, nullptr, nullptr, nullptr, nullptr, 1, 0, 0, block_n, stream, &r);
}

GROMA_API int32_t groma_splitk_reduce(const float* ws, int32_t splits, int32_t M, int32_t N, int32_t act,
                                       int32_t flags, const float* bias, const float* gamma, const void* residual,
                                       void* out, int64_t ld_m, int64_t ld_n, void* stream) {
    if (!ws || !out || splits < 1 || M <= 0 || N <= 0) return GROMA_ERR_ARG;
    const long long total = (long long)M * N;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    splitk_reduce_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        ws, splits, M, N, act, flags, bias, gamma, reinterpret_cast<const __nv_bfloat16*>(residual), out, ld_m, ld_n);
    return cudaGetLastError() == cudaSuccess ? GROMA_OK : GROMA_ERR_CUDA;
}
