// Fused softmax(QK^T*scale + mask) V for bf16, head dims 32/64/128: online-softmax tiles of 64 queries x 64 keys,
// cp.async double-buffered K/V, ldmatrix + mma.sync.m16n8k16 (fp32 accumulate), causal / per-batch key-length masks.
// Serves: LLaMA prefill + decode (modeling_llama.py:199-289 semantics), DINOv2 global attention
// (modeling_dinov2.py:153-179) and the DDETR decoder self-attention (modeling_deformable_detr.py:453-516).
#include "ptx.cuh"
#include "decode_common.cuh"
#include "capi_common.h"
#include <cooperative_groups.h>

namespace gb {

struct AttnParams {
    const __nv_bfloat16* q; long long q_bs, q_rs;   // q[b*q_bs + i*q_rs + h*D + d]
    const __nv_bfloat16* k; long long k_bs, k_hs, k_rs;  // k[b*k_bs + h*k_hs + j*k_rs + d]
    const __nv_bfloat16* v; long long v_bs, v_hs, v_rs;
    __nv_bfloat16* o; long long o_bs, o_rs;          // o[b*o_bs + i*o_rs + h*D + d]
    const int* kv_len;                               // optional [B]: keys >= kv_len[b] are masked
    int Sq, Sk, H;
    int q_pos0;      // causal: key j visible to query i iff j <= q_pos0 + i
    float scale_log2;  // softmax scale * log2(e)
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

constexpr int ATT_BM = 64, ATT_BN = 64, ATT_THREADS = 128;

template <int D, bool CAUSAL>
__global__ void __launch_bounds__(ATT_THREADS) attention_kernel(const AttnParams p) {
    constexpr int LDS = D + 8;           // padded smem row (elements)
    constexpr int CHUNKS = D / 8;        // 16-byte chunks per row
    extern __shared__ __align__(16) uint8_t smem_att[];
    __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(smem_att);
    __nv_bfloat16* Ks = Qs + ATT_BM * LDS;       // [2][BN][LDS]
    __nv_bfloat16* Vs = Ks + 2 * ATT_BN * LDS;   // [2][BN][LDS]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int q0 = qt * ATT_BM;
    int sk = p.Sk;
    if (p.kv_len) sk = min(sk, p.kv_len[b]);
    int k_end = sk;
    if (CAUSAL) k_end = min(sk, p.q_pos0 + min(q0 + ATT_BM, p.Sq));
    const int n_blocks = (k_end + ATT_BN - 1) / ATT_BN;

    const __nv_bfloat16* qg = p.q + (long long)b * p.q_bs + (long long)h * D;
    const __nv_bfloat16* kg = p.k + (long long)b * p.k_bs + (long long)h * p.k_hs;
    const __nv_bfloat16* vg = p.v + (long long)b * p.v_bs + (long long)h * p.v_hs;

    // ---- async load of Q tile and first K/V block
    for (int c = tid; c < ATT_BM * CHUNKS; c += ATT_THREADS) {
        const int r = c / CHUNKS, ch = c % CHUNKS;
        const bool ok = q0 + r < p.Sq;
        cp_async16(Qs + r * LDS + ch * 8, qg + (long long)(ok ? q0 + r : 0) * p.q_rs + ch * 8, ok);
    }
    auto load_kv = [&](int blk, int buf) {
        const int j0 = blk * ATT_BN;
        for (int c = tid; c < ATT_BN * CHUNKS; c += ATT_THREADS) {
            const int r = c / CHUNKS, ch = c % CHUNKS;
            const bool ok = j0 + r < sk;
            const long long row = ok ? j0 + r : 0;
            cp_async16(Ks + (buf * ATT_BN + r) * LDS + ch * 8, kg + row * p.k_rs + ch * 8, ok);
            cp_async16(Vs + (buf * ATT_BN + r) * LDS + ch * 8, vg + row * p.v_rs + ch * 8, ok);
        }
    };
    if (n_blocks > 0) load_kv(0, 0);
    cp_async_commit();

    float acc_o[D / 8][4];
#pragma unroll
    for (int i = 0; i < D / 8; ++i) { acc_o[i][0] = acc_o[i][1] = acc_o[i][2] = acc_o[i][3] = 0.f; }
    float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};
    uint32_t qf[D / 16][4];

    const int row_in_warp0 = lane >> 2;              // accumulator rows: row_in_warp0 and +8
    const int qrow0 = q0 + warp * 16 + row_in_warp0;  // global query index of c0/c1 ; +8 for c2/c3

    for (int blk = 0; blk < n_blocks; ++blk) {
        const int buf = blk & 1;
        if (blk + 1 < n_blocks) load_kv(blk + 1, buf ^ 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        if (blk == 0) {
#pragma unroll
            for (int ks = 0; ks < D / 16; ++ks) {
                const uint32_t addr = smem_u32(Qs + (warp * 16 + (lane & 15)) * LDS + ks * 16 + (lane >> 4) * 8);
                ldsm_x4(addr, qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
            }
        }
        // ---- S = Q K^T  (16 x 64 per warp)
        float s[ATT_BN / 8][4];
#pragma unroll
        for (int i = 0; i < ATT_BN / 8; ++i) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f; }
        const __nv_bfloat16* kb = Ks + buf * ATT_BN * LDS;
#pragma unroll
        for (int ks = 0; ks < D / 16; ++ks) {
#pragma unroll
            for (int np = 0; np < ATT_BN / 16; ++np) {
                uint32_t b0, b1, b2, b3;
                const int n = np * 16 + (lane >> 4) * 8 + (lane & 7);
                const int kk = ks * 16 + ((lane >> 3) & 1) * 8;
                ldsm_x4(smem_u32(kb + n * LDS + kk), b0, b1, b2, b3);
                mma_bf16_16816(s[2 * np], qf[ks], b0, b1);
                mma_bf16_16816(s[2 * np + 1], qf[ks], b2, b3);
            }
        }
        // ---- mask + online softmax
        const int j_base = blk * ATT_BN + (lane & 3) * 2;
        float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int nt = 0; nt < ATT_BN / 8; ++nt) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = j_base + nt * 8 + (e & 1);
                const int qi = qrow0 + (e >> 1) * 8;
                bool ok = j < sk;
                if (CAUSAL) ok = ok && (j <= p.q_pos0 + qi);
                const float x = ok ? s[nt][e] * p.scale_log2 : -INFINITY;
                s[nt][e] = x;
                mx[e >> 1] = fmaxf(mx[e >> 1], x);
            }
        }
        float corr[2], m_safe[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
            mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
            const float m_new = fmaxf(m_run[r], mx[r]);
            m_safe[r] = (m_new == -INFINITY) ? 0.f : m_new;
            corr[r] = exp2f(m_run[r] - m_safe[r]);  // m_run = -inf -> 0
            m_run[r] = m_new;
        }
        float rs[2] = {0.f, 0.f};
        uint32_t pf[ATT_BN / 16][4];
#pragma unroll
        for (int nt = 0; nt < ATT_BN / 8; ++nt) {
            const float p0 = exp2f(s[nt][0] - m_safe[0]);
            const float p1 = exp2f(s[nt][1] - m_safe[0]);
            const float p2 = exp2f(s[nt][2] - m_safe[1]);
            const float p3 = exp2f(s[nt][3] - m_safe[1]);
            rs[0] += p0 + p1;
            rs[1] += p2 + p3;
            pf[nt >> 1][(nt & 1) * 2 + 0] = pack_bf16x2(p0, p1);
            pf[nt >> 1][(nt & 1) * 2 + 1] = pack_bf16x2(p2, p3);
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) l_run[r] = l_run[r] * corr[r] + rs[r];
#pragma unroll
        for (int dt = 0; dt < D / 8; ++dt) {
            acc_o[dt][0] *= corr[0]; acc_o[dt][1] *= corr[0];
            acc_o[dt][2] *= corr[1]; acc_o[dt][3] *= corr[1];
        }
        // ---- O += P V
        const __nv_bfloat16* vb = Vs + buf * ATT_BN * LDS;
#pragma unroll
        for (int kt = 0; kt < ATT_BN / 16; ++kt) {
#pragma unroll
            for (int dp = 0; dp < D / 16; ++dp) {
                uint32_t b0, b1, b2, b3;
                const int kr = kt * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
                const int dc = dp * 16 + (lane >> 4) * 8;
                ldsm_x4_t(smem_u32(vb + kr * LDS + dc), b0, b1, b2, b3);
                mma_bf16_16816(acc_o[2 * dp], pf[kt], b0, b1);
                mma_bf16_16816(acc_o[2 * dp + 1], pf[kt], b2, b3);
            }
        }
        __syncthreads();  // everyone done with buf before it is refilled two iterations later
    }
    cp_async_wait<0>();

    // ---- finalize: O /= l
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 1);
        l_run[r] += __shfl_xor_sync(0xffffffffu, l_run[r], 2);
    }
    const float inv0 = l_run[0] > 0.f ? 1.f / l_run[0] : 0.f;
    const float inv1 = l_run[1] > 0.f ? 1.f / l_run[1] : 0.f;
    __nv_bfloat16* og = p.o + (long long)b * p.o_bs + (long long)h * D;
#pragma unroll
    for (int dt = 0; dt < D / 8; ++dt) {
        const int d = dt * 8 + (lane & 3) * 2;
        if (qrow0 < p.Sq)
            *reinterpret_cast<uint32_t*>(og + (long long)qrow0 * p.o_rs + d) = pack_bf16x2(acc_o[dt][0] * inv0, acc_o[dt][1] * inv0);
        if (qrow0 + 8 < p.Sq)
            *reinterpret_cast<uint32_t*>(og + (long long)(qrow0 + 8) * p.o_rs + d) = pack_bf16x2(acc_o[dt][2] * inv1, acc_o[dt][3] * inv1);
    }
}

template <int D, bool CAUSAL>
static int launch_attn(const AttnParams& p, int B, cudaStream_t st) {
    constexpr int SMEM = (ATT_BM + 4 * ATT_BN) * (D + 8) * 2;
    static bool set = false;
    if (!set) {
        if (cudaFuncSetAttribute(attention_kernel<D, CAUSAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) != cudaSuccess)
            return GROMA_ERR_CUDA;
        set = true;
    }
    dim3 grid((p.Sq + ATT_BM - 1) / ATT_BM, p.H, B);
    attention_kernel<D, CAUSAL><<<grid, ATT_THREADS, SMEM, st>>>(p);
    return GROMA_LAUNCH_CHECK();
}

}  // namespace gb
using namespace gb;

GROMA_API int32_t groma_attention(const void* q, int64_t q_bs, int64_t q_rs, const void* k, int64_t k_bs, int64_t k_hs,
                                  int64_t k_rs, const void* v, int64_t v_bs, int64_t v_hs, int64_t v_rs, void* o,
                                  int64_t o_bs, int64_t o_rs, const int32_t* kv_len, int32_t B, int32_t H, int32_t Sq,
                                  int32_t Sk, int32_t D, int32_t causal, int32_t q_pos0, float scale, void* stream) {
    if (!q || !k || !v || !o || B <= 0 || H <= 0 || Sq <= 0 || Sk <= 0) return GROMA_ERR_ARG;
    if ((q_rs & 7) || (k_rs & 7) || (v_rs & 7) || (o_rs & 1) || (q_bs & 7) || (k_bs & 7) || (k_hs & 7) || (v_bs & 7) || (v_hs & 7))
        return GROMA_ERR_ALIGN;
    AttnParams p;
    p.q = reinterpret_cast<const __nv_bfloat16*>(q); p.q_bs = q_bs; p.q_rs = q_rs;
    p.k = reinterpret_cast<const __nv_bfloat16*>(k); p.k_bs = k_bs; p.k_hs = k_hs; p.k_rs = k_rs;
    p.v = reinterpret_cast<const __nv_bfloat16*>(v); p.v_bs = v_bs; p.v_hs = v_hs; p.v_rs = v_rs;
    p.o = reinterpret_cast<__nv_bfloat16*>(o); p.o_bs = o_bs; p.o_rs = o_rs;
    p.kv_len = kv_len; p.Sq = Sq; p.Sk = Sk; p.H = H; p.q_pos0 = q_pos0;
    p.scale_log2 = scale * 1.4426950408889634f;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (D == 128) return causal ? launch_attn<128, true>(p, B, st) : launch_attn<128, false>(p, B, st);
    if (D == 64) return causal ? launch_attn<64, true>(p, B, st) : launch_attn<64, false>(p, B, st);
    if (D == 32) return causal ? launch_attn<32, true>(p, B, st) : launch_attn<32, false>(p, B, st);
    return GROMA_ERR_UNSUPPORTED;
}

// ------------------------------------------------------------------------------------------------------------------
// Decode attention (one query token per sequence): HBM-bound streaming of the K/V cache, no tensor cores.
// Semantics = groma/model/groma.py:376-379 + eager LLaMA attention: every cached position < kv_len[b] is visible.
// One 2-CTA cluster per (head, batch row), the keys split between the pair.  Per CTA one producer lane issues 1-D bulk copies
// of DT_KEYS consecutive K rows and V rows (contiguous in the [B,H,cap,D] cache) into a DT_STAGES-deep shared-memory ring;
// the DEC_WARPS consumer warps cover two keys per warp and step (16 lanes x 16 bytes = one 256-byte row per half-warp), fold
// DT_UNROLL steps into each online-softmax update, and merge their half-warp states through shared memory, then the pair's
// states through distributed shared memory.  Bytes in flight do not depend on registers/occupancy: 8 resident CTAs x 24 KB
// per SM.
namespace gb {

#ifndef GROMA_DEC_WARPS
#define GROMA_DEC_WARPS 2
#endif
#ifndef GROMA_DEC_SPLIT
#define GROMA_DEC_SPLIT 2
#endif
constexpr int DEC_WARPS = GROMA_DEC_WARPS;   // 2 warps/CTA, 2 CTAs (one cluster) per (batch, head): 2*B*H CTAs all resident in one wave
constexpr int DEC_SPLIT = GROMA_DEC_SPLIT;                   // keys are split over the CTAs of a cluster; partials merge through DSMEM

constexpr int DT_UNROLL = 4;
constexpr int DT_KEYS = DEC_WARPS * 2 * DT_UNROLL;   // keys per stage (16)
#ifndef GROMA_DT_STAGES
#define GROMA_DT_STAGES 2
#endif
constexpr int DT_STAGES = GROMA_DT_STAGES;

// ROPE = true additionally folds the kernel in front of it into the prologue (one launch less per layer): q, and the new
// token's K/V row, are reduced from the qkv GEMM's split-K partials ws[S][B][3*H*D] and rotated exactly as
// reduce_rope_kv_kernel does (shared code in decode_common.cuh); the CTA whose key range holds position *pos_ptr writes the
// new K/V row into the cache and substitutes it for the (stale) staged copy when that key comes up, so the key order -- and
// every bit of the result -- is that of reduce_rope_kv_kernel followed by the ROPE = false kernel.
struct DecodeRopeArgs {
    const float* ws; int S;
    const float* cos_t; const float* sin_t;
    const int* pos_ptr;
};

template <int D, bool ROPE>
__global__ void __cluster_dims__(DEC_SPLIT, 1, 1) __launch_bounds__((DEC_WARPS + 1) * 32) decode_attention_tma_kernel(
    const __nv_bfloat16* __restrict__ q, __nv_bfloat16* __restrict__ kc, __nv_bfloat16* __restrict__ vc,
    __nv_bfloat16* __restrict__ out, const int* __restrict__ kv_len, int H, long long cap, float scale_log2, DecodeRopeArgs ra) {
    static_assert(D == 128, "16 lanes x 8 dims");
    static_assert(!ROPE || DEC_WARPS * 32 == D / 2, "one consumer thread per rotary pair");
    __shared__ __align__(16) __nv_bfloat16 s_new[3][D];   // ROPE: q, new k row, new v row
    __shared__ __align__(128) __nv_bfloat16 ring[DT_STAGES][2][DT_KEYS * D];
    __shared__ __align__(8) uint64_t full_bar[DT_STAGES], empty_bar[DT_STAGES];
    __shared__ float sm_m[DEC_WARPS * 2], sm_l[DEC_WARPS * 2], sm_acc[DEC_WARPS * 2][D];
    __shared__ float peer_m[DEC_SPLIT], peer_l[DEC_SPLIT], peer_acc[DEC_SPLIT][D];
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // distributed-shared-memory rule: a CTA may only touch a peer's shared memory once that peer is known to be running.
    // Arrive now, wait just before the first remote store -- the barrier latency hides behind the key loop.
    cluster_arrive_relaxed();
    if (threadIdx.x == 0) {
        for (int s = 0; s < DT_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], DEC_WARPS); }
        fence_barrier_init();
    }
    __syncthreads();
    asm volatile("griddepcontrol.wait;" ::: "memory");
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int crank = (int)cluster.block_rank();
    const int h = blockIdx.x / DEC_SPLIT, b = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int grp = lane >> 4, l = lane & 15;
    const int n_all = kv_len[b];
    const int per = (n_all + DEC_SPLIT - 1) / DEC_SPLIT;
    const int k_begin = min(crank * per, n_all);
    const int n = min(n_all, k_begin + per) - k_begin;
    const int nchunks = (n + DT_KEYS - 1) / DT_KEYS;
    __nv_bfloat16* kb = kc + (((long long)b * H + h) * cap + k_begin) * D;
    __nv_bfloat16* vb = vc + (((long long)b * H + h) * cap + k_begin) * D;
    int newidx = -1;          // ROPE: index (within this CTA's key range) of the token appended by this step, if it is ours
    bool append = false;      // ROPE: this CTA writes the new K/V row (the range owner; the last CTA if no range holds it)
    if constexpr (ROPE) {
        const int pos = *ra.pos_ptr;
        if (pos >= k_begin && pos < k_begin + n) newidx = pos - k_begin;
        append = newidx >= 0 || (pos >= n_all && crank == DEC_SPLIT - 1);
    }
    if (warp == DEC_WARPS) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int c = 0; c < nchunks; ++c) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                const int keys = min(DT_KEYS, n - c * DT_KEYS);
                const uint32_t bytes = (uint32_t)keys * D * 2;
                mbar_expect_tx(&full_bar[stage], 2 * bytes);
                bulk_load_1d(&ring[stage][0][0], kb + (long long)c * DT_KEYS * D, bytes, &full_bar[stage]);
                bulk_load_1d(&ring[stage][1][0], vb + (long long)c * DT_KEYS * D, bytes, &full_bar[stage]);
                if (++stage == DT_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        float qf[8];
        if constexpr (ROPE) {
            constexpr int half = D / 2;
            const int j = threadIdx.x;                       // one rotary pair (j, j + half) per consumer thread
            const int N = 3 * H * D;
            // every partial of q (and k, v in the appending CTA) is in flight before the first add, and behind the position load:
            // the prologue costs two L2 round trips (pos -> cos/sin) instead of 1 + S (+ 2S)
            const int pos = *ra.pos_ptr;
            const int cols[3] = {h * D, H * D + h * D, 2 * H * D + h * D};
            float s1[3], s2[3];
            if (append) {
                splitk_pairs<3>(ra.ws, ra.S, (int)gridDim.y, N, b, cols, j, half, s1, s2);
            } else {
                const int c0[1] = {cols[0]};
                float t1[1], t2[1];
                splitk_pairs<1>(ra.ws, ra.S, (int)gridDim.y, N, b, c0, j, half, t1, t2);
                s1[0] = t1[0]; s2[0] = t2[0];
            }
            const float c = ra.cos_t[(long long)pos * half + j], sn = ra.sin_t[(long long)pos * half + j];
            float q1 = s1[0], q2 = s2[0];
            q1 = bf16_round(q1); q2 = bf16_round(q2);
            rope_pair(q1, q2, c, sn, s_new[0][j], s_new[0][j + half]);
            if (append) {
                float k1 = s1[1], k2 = s2[1];
                const float v1 = s1[2], v2 = s2[2];
                k1 = bf16_round(k1); k2 = bf16_round(k2);
                rope_pair(k1, k2, c, sn, s_new[1][j], s_new[1][j + half]);
                s_new[2][j] = __float2bfloat16_rn(v1);
                s_new[2][j + half] = __float2bfloat16_rn(v2);
                __nv_bfloat16* kn = kc + (((long long)b * H + h) * cap + pos) * D;   // append to the cache for the following steps
                __nv_bfloat16* vn = vc + (((long long)b * H + h) * cap + pos) * D;
                kn[j] = s_new[1][j]; kn[j + half] = s_new[1][j + half];
                vn[j] = s_new[2][j]; vn[j + half] = s_new[2][j + half];
            }
            asm volatile("bar.sync 1, %0;" ::"n"(DEC_WARPS * 32) : "memory");   // consumer warps only
        }
        {
            const uint4 qv = ROPE ? *reinterpret_cast<const uint4*>(&s_new[0][l * 8])
                                  : *reinterpret_cast<const uint4*>(q + ((long long)b * H + h) * D + l * 8);
            const __nv_bfloat162* q2 = reinterpret_cast<const __nv_bfloat162*>(&qv);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const float2 f = __bfloat1622float2(q2[t]);
                qf[2 * t] = f.x * scale_log2;
                qf[2 * t + 1] = f.y * scale_log2;
            }
        }
        float m = -INFINITY, lsum = 0.f, acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        constexpr int STEP = DEC_WARPS * 2;
        const int slot = warp * 2 + grp;
        int stage = 0;
        uint32_t phase = 0;
        for (int c = 0; c < nchunks; ++c) {
            mbar_wait(&full_bar[stage], phase);
            const __nv_bfloat16* ks = &ring[stage][0][0];
            const __nv_bfloat16* vs = &ring[stage][1][0];
            const int left = n - c * DT_KEYS;   // valid keys in this stage
            float s[DT_UNROLL];
            uint4 vv[DT_UNROLL];
#pragma unroll
            for (int u = 0; u < DT_UNROLL; ++u) {
                const int j = slot + u * STEP;
                const bool ok = j < left;
                uint4 kk = ok ? *reinterpret_cast<const uint4*>(ks + j * D + l * 8) : make_uint4(0, 0, 0, 0);
                vv[u] = ok ? *reinterpret_cast<const uint4*>(vs + j * D + l * 8) : make_uint4(0, 0, 0, 0);
                if (ROPE && c * DT_KEYS + j == newidx) {     // this step's token: its staged copy predates the append
                    kk = *reinterpret_cast<const uint4*>(&s_new[1][l * 8]);
                    vv[u] = *reinterpret_cast<const uint4*>(&s_new[2][l * 8]);
                }
                const __nv_bfloat162* k2 = reinterpret_cast<const __nv_bfloat162*>(&kk);
                float d = 0.f;
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float2 f = __bfloat1622float2(k2[t]);
                    d += f.x * qf[2 * t] + f.y * qf[2 * t + 1];
                }
                d += __shfl_xor_sync(0xffffffffu, d, 8);
                d += __shfl_xor_sync(0xffffffffu, d, 4);
                d += __shfl_xor_sync(0xffffffffu, d, 2);
                d += __shfl_xor_sync(0xffffffffu, d, 1);
                s[u] = ok ? d : -INFINITY;
            }
            float mn = m;
#pragma unroll
            for (int u = 0; u < DT_UNROLL; ++u) mn = fmaxf(mn, s[u]);
            const float mref = (mn == -INFINITY) ? 0.f : mn;
            const float corr = exp2f(m - mref);
            m = mn;
            lsum *= corr;
#pragma unroll
            for (int t = 0; t < 8; ++t) acc[t] *= corr;
#pragma unroll
            for (int u = 0; u < DT_UNROLL; ++u) {
                const float p = exp2f(s[u] - mref);
                lsum += p;
                const float pr = bf16_round(p);
                const __nv_bfloat162* v2 = reinterpret_cast<const __nv_bfloat162*>(&vv[u]);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float2 f = __bfloat1622float2(v2[t]);
                    acc[2 * t] += pr * f.x;
                    acc[2 * t + 1] += pr * f.y;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty_bar[stage]);
            if (++stage == DT_STAGES) { stage = 0; phase ^= 1; }
        }
        if (l == 0) { sm_m[slot] = m; sm_l[slot] = lsum; }
#pragma unroll
        for (int t = 0; t < 8; ++t) sm_acc[slot][l * 8 + t] = acc[t];
    }
    __syncthreads();
    cluster_wait();
    float* r_m = cluster.map_shared_rank(peer_m, 0);
    float* r_l = cluster.map_shared_rank(peer_l, 0);
    float* r_acc = cluster.map_shared_rank(&peer_acc[0][0], 0);
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float M = -INFINITY;
#pragma unroll
        for (int w = 0; w < DEC_WARPS * 2; ++w) M = fmaxf(M, sm_m[w]);
        float num = 0.f, den = 0.f;
#pragma unroll
        for (int w = 0; w < DEC_WARPS * 2; ++w) {
            const float c = (sm_m[w] == -INFINITY) ? 0.f : exp2f(sm_m[w] - M);
            num += c * sm_acc[w][d];
            den += c * sm_l[w];
        }
        r_acc[crank * D + d] = num;
        if (d == 0) { r_m[crank] = M; r_l[crank] = den; }
    }
    cluster.sync();
    if (crank == 0) {
        for (int d = threadIdx.x; d < D; d += blockDim.x) {
            float M = -INFINITY;
#pragma unroll
            for (int r = 0; r < DEC_SPLIT; ++r) M = fmaxf(M, peer_m[r]);
            float num = 0.f, den = 0.f;
#pragma unroll
            for (int r = 0; r < DEC_SPLIT; ++r) {
                const float c = (peer_m[r] == -INFINITY) ? 0.f : exp2f(peer_m[r] - M);
                num += c * peer_acc[r][d];
                den += c * peer_l[r];
            }
            out[((long long)b * H + h) * D + d] = __float2bfloat16_rn(den > 0.f ? num / den : 0.f);
        }
    }
}

}  // namespace gb

GROMA_API int32_t groma_decode_attention(const void* q, const void* cache_k, const void* cache_v, void* out,
                                         const int32_t* kv_len, int32_t B, int32_t H, int32_t D, int64_t cap, float scale,
                                         int32_t pdl, void* stream) {
    if (!q || !cache_k || !cache_v || !out || !kv_len || B <= 0 || H <= 0) return GROMA_ERR_ARG;
    if (D != 128) return GROMA_ERR_UNSUPPORTED;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(H * gb::DEC_SPLIT, B); cfg.blockDim = dim3((gb::DEC_WARPS + 1) * 32); cfg.dynamicSmemBytes = 0;
    cfg.stream = reinterpret_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    if (pdl) { cfg.attrs = attr; cfg.numAttrs = 1; }
    cudaError_t e = cudaLaunchKernelEx(&cfg, gb::decode_attention_tma_kernel<128, false>, reinterpret_cast<const __nv_bfloat16*>(q),
                                       reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(cache_k)),
                                       reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(cache_v)),
                                       reinterpret_cast<__nv_bfloat16*>(out), kv_len, (int)H, (long long)cap,
                                       scale * 1.4426950408889634f, gb::DecodeRopeArgs{});
    return e == cudaSuccess ? GROMA_OK : GROMA_ERR_CUDA;
}

GROMA_API int32_t groma_decode_rope_attention(const float* ws, int32_t splits, void* cache_k, void* cache_v, void* out,
                                              const int32_t* kv_len, const int32_t* pos_ptr, const float* cos_t, const float* sin_t,
                                              int32_t B, int32_t H, int32_t D, int64_t cap, float scale, int32_t pdl, void* stream) {
    if (!ws || !cache_k || !cache_v || !out || !kv_len || !pos_ptr || !cos_t || !sin_t || B <= 0 || H <= 0 || splits < 1) return GROMA_ERR_ARG;
    if (D != 128) return GROMA_ERR_UNSUPPORTED;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(H * gb::DEC_SPLIT, B); cfg.blockDim = dim3((gb::DEC_WARPS + 1) * 32); cfg.dynamicSmemBytes = 0;
    cfg.stream = reinterpret_cast<cudaStream_t>(stream);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    if (pdl) { cfg.attrs = attr; cfg.numAttrs = 1; }
    gb::DecodeRopeArgs ra{ws, splits, cos_t, sin_t, pos_ptr};
    cudaError_t e = cudaLaunchKernelEx(&cfg, gb::decode_attention_tma_kernel<128, true>, (const __nv_bfloat16*)nullptr,
                                       reinterpret_cast<__nv_bfloat16*>(cache_k), reinterpret_cast<__nv_bfloat16*>(cache_v),
                                       reinterpret_cast<__nv_bfloat16*>(out), kv_len, (int)H, (long long)cap,
                                       scale * 1.4426950408889634f, ra);
    return e == cudaSuccess ? GROMA_OK : GROMA_ERR_CUDA;
}
